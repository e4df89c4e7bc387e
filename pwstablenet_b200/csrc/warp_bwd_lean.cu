// warp_bwd_lean.cu -- backward warp specialised for the reference's hot layouts
// (NCHW frames / grad_output W-contiguous, map planar or interleaved, C in {1,3}).
//
// Same algorithm as the generic marching kernel in warp_bwd.cu (horizontal take-over of the
// east taps by shuffle, vertical carry of the south taps in registers, one RED per source
// pixel and channel in the regular case) with the costs the first profile showed removed:
// padding / align_corners are template flags, row pointers are advanced instead of
// recomputed, and a warp whose 32 pixels have all four taps inside the frame runs a
// mask-free body.  Autograd of R/main_new.py:106,116 (grad -> map) and :197 (grad -> frame).
#include "pws_tile.cuh"

namespace pws {

namespace {

constexpr int kRows = 8, kWarpsX = 2, kWarpsY = 4;
constexpr int kThreads = 32 * kWarpsX * kWarpsY;
constexpr int kTW = 32 * kWarpsX, kTH = kRows * kWarpsY;

template <int CS>
struct Carry {
    int x, y;     // target of the parked south-west sums
    bool live;
    float v[CS];
};

// One output row of a warp.  kMasked=false: every lane is a real pixel with 4 valid taps.
template <typename T, typename G, int CS, bool kGin, bool kGgrid, bool kMasked>
__device__ __forceinline__ void row_body(
    const int lane, const bool px_ok, const unsigned live,
    const float ix, const float iy, const float gxm, const float gym, const float (&go)[CS],
    const T *__restrict__ ip, const int sH, const int i_ch, const int H, const int W,
    float *__restrict__ gip, const int gi_ch,
    G *__restrict__ ggq, const int gg_s3, Carry<CS> &cy, int2 *__restrict__ queue)
{
    const float x0f = floorf(ix), y0f = floorf(iy);
    const int x0 = (int)x0f, y0 = (int)y0f;
    const float dw = fsub(x0f + 1.0f, ix), de = fsub(ix, x0f), dn = fsub(y0f + 1.0f, iy), ds = fsub(iy, y0f);
    unsigned mask = 15u;
    if (kMasked) {
        const bool xw = (unsigned)x0 < (unsigned)W, xe = (unsigned)(x0 + 1) < (unsigned)W;
        const bool yn = (unsigned)y0 < (unsigned)H, ys = (unsigned)(y0 + 1) < (unsigned)H;
        mask = ((xw && yn) ? 1u : 0u) | ((xe && yn) ? 2u : 0u) | ((xw && ys) ? 4u : 0u) | ((xe && ys) ? 8u : 0u);
        if (!px_ok) mask = 0u;
    }
    const int o_nw = y0 * sH + x0;  // same offset in the frame and in grad_input (both W-contiguous, pitch sH == W)

    if (kGgrid && (!kMasked || px_ok)) {
        float gix = 0.f, giy = 0.f;
#pragma unroll
        for (int k = 0; k < CS; ++k) {
            const T *__restrict__ pc = ip + (k * i_ch + o_nw);
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
            if (!kMasked || (mask & 1u)) v0 = to_acc(ldg(pc));
            if (!kMasked || (mask & 2u)) v1 = to_acc(ldg(pc + 1));
            if (!kMasked || (mask & 4u)) v2 = to_acc(ldg(pc + sH));
            if (!kMasked || (mask & 8u)) v3 = to_acc(ldg(pc + sH + 1));
            // ATen's statement order: t = v*d rounded, then one fma with gOut
            if (!kMasked || (mask & 1u)) { gix = ffma(-fmul(v0, dn), go[k], gix); giy = ffma(-fmul(v0, dw), go[k], giy); }
            if (!kMasked || (mask & 2u)) { gix = ffma(fmul(v1, dn), go[k], gix);  giy = ffma(-fmul(v1, de), go[k], giy); }
            if (!kMasked || (mask & 4u)) { gix = ffma(-fmul(v2, ds), go[k], gix); giy = ffma(fmul(v2, dw), go[k], giy); }
            if (!kMasked || (mask & 8u)) { gix = ffma(fmul(v3, ds), go[k], gix);  giy = ffma(fmul(v3, de), go[k], giy); }
        }
        gix = fmul(gxm, gix); giy = fmul(gym, giy);
        if (gg_s3 == 1) st_pair(ggq, gix, giy);
        else { ggq[0] = from_acc<G, float>(gix); ggq[gg_s3] = from_acc<G, float>(giy); }
    }

    if (kGin) {
        const float nw = fmul(dw, dn), ne = fmul(de, dn), sw = fmul(dw, ds), se = fmul(de, ds);
        const int px0 = __shfl_up_sync(0xffffffffu, x0, 1), py0 = __shfl_up_sync(0xffffffffu, y0, 1);
        const int nx0 = __shfl_down_sync(0xffffffffu, x0, 1), ny0 = __shfl_down_sync(0xffffffffu, y0, 1);
        bool take = lane > 0 && px0 + 1 == x0 && py0 == y0;
        bool given = lane < 31 && nx0 == x0 + 1 && ny0 == y0;
        if (kMasked) {
            take = take && px_ok && ((live >> (lane - 1)) & 1u);
            given = given && px_ok && ((live >> (lane + 1)) & 1u);
        }
        const bool chain = cy.live && cy.x == x0 && cy.y == y0;
        const int o_cy = cy.y * sH + cy.x;
        // Left-overs -- east taps nobody takes over, parked south sums whose chain broke -- exist on a
        // few lanes of almost every row of a stretched map.  The L2 accepts ~25 G RED instructions/s
        // whether 1 or 32 lanes are active (tools/exp/exp_red.cu), and issuing them per class made the
        // scatter run exactly at that ceiling (9 of 12 REDs per row).  They are compacted through a
        // small per-warp queue in shared memory instead and leave as one dense RED.
        const bool p_e1 = !given && (mask & 2u), p_e2 = !given && (mask & 8u), p_f = cy.live && !chain;
        const unsigned b_e1 = __ballot_sync(0xffffffffu, p_e1), b_e2 = __ballot_sync(0xffffffffu, p_e2);
        const unsigned b_f = __ballot_sync(0xffffffffu, p_f);
        const unsigned lt = (1u << lane) - 1u;
        const int n_e1 = __popc(b_e1), n_e2 = __popc(b_e2), n_f = __popc(b_f);
        const int s_e1 = __popc(b_e1 & lt), s_e2 = CS * n_e1 + __popc(b_e2 & lt), s_f = CS * (n_e1 + n_e2) + __popc(b_f & lt);
#pragma unroll
        for (int k = 0; k < CS; ++k) {
            float top = fmul(nw, go[k]), bot = fmul(sw, go[k]);
            const float etop = fmul(ne, go[k]), ebot = fmul(se, go[k]);
            const float ptop = __shfl_up_sync(0xffffffffu, etop, 1), pbot = __shfl_up_sync(0xffffffffu, ebot, 1);
            if (take) { top += ptop; bot += pbot; }
            if (p_e1) queue[s_e1 + k * n_e1] = make_int2(k * gi_ch + o_nw + 1, __float_as_int(etop));
            if (p_e2) queue[s_e2 + k * n_e2] = make_int2(k * gi_ch + o_nw + sH + 1, __float_as_int(ebot));
            if (chain) top += cy.v[k];
            if (p_f) queue[s_f + k * n_f] = make_int2(k * gi_ch + o_cy, __float_as_int(cy.v[k]));
            if (mask & 1u) atomicAdd(gip + (k * gi_ch + o_nw), top);
            cy.v[k] = bot;
        }
        const int n_items = CS * (n_e1 + n_e2 + n_f);
        if (n_items > 0) {
            __syncwarp();
            for (int i = lane; i < n_items; i += 32) {
                const int2 it = queue[i];
                atomicAdd(gip + it.x, __int_as_float(it.y));
            }
            __syncwarp();
        }
        cy.x = x0; cy.y = y0 + 1;
        cy.live = (mask & 4u) != 0u;
    }
}

// T: element type of the frame and of grad_output (float, __half or __nv_bfloat16).  G: element type of the map and of
// grad_grid (float, or T for 16-bit frames).  The arithmetic and the grad_input accumulation buffer are fp32 whatever T and
// G are; grad_grid is rounded to G once, at its store.
template <typename T, typename G, int CS, bool kBorder, bool kAlign, bool kGin, bool kGgrid>
#ifndef PWS_BWD_MINB
#define PWS_BWD_MINB 4   // 64 registers, 32 warps/SM: measured 5-9 % faster than 3 CTAs at 80 registers
#endif
__global__ void __launch_bounds__(kThreads, PWS_BWD_MINB)
bwd_lean_kernel(const View gout, const View in, const View grid, const View gin, const View ggrid,
                const Geometry g, const int n_begin)
{
    __shared__ int2 s_queue[kGin ? kThreads / 32 : 1][kGin ? 3 * CS * 32 : 1];  // per warp: every lane, 3 classes, CS channels
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    int2 *const queue = s_queue[kGin ? wrp : 0];
    const int n = n_begin + blockIdx.z;
    const int w = blockIdx.x * kTW + (wrp % kWarpsX) * 32 + lane;
    const int h0 = blockIdx.y * kTH + (wrp / kWarpsX) * kRows;
    if (h0 >= g.Ho) return;  // warp-uniform
    const bool col_ok = w < g.Wo;
    const unsigned live = __ballot_sync(0xffffffffu, col_ok);
    const int rows = min(kRows, g.Ho - h0);
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);

    const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
    float *__restrict__ gip = kGin ? (float *)gin.p + (int64_t)n * gin.sN : nullptr;
    const int sH = in.s2;
    const int i_ch = in.s1, gi_ch = kGin ? gin.s1 : 0, go_ch = gout.s1;  // 32-bit in-frame offsets (validated on the host)

    const bool inter = grid.s3 == 1;
    const G *__restrict__ gq = (const G *)grid.p + (int64_t)n * grid.sN + (int64_t)h0 * grid.s1 + (int64_t)w * grid.s2;
    const T *__restrict__ goq = (const T *)gout.p + (int64_t)n * gout.sN + (int64_t)h0 * gout.s2 + w;
    G *__restrict__ ggq = kGgrid ? (G *)ggrid.p + (int64_t)n * ggrid.sN + (int64_t)h0 * ggrid.s1 + (int64_t)w * ggrid.s2 : nullptr;

    Carry<CS> cy;
    cy.x = 0; cy.y = 0; cy.live = false;
#pragma unroll
    for (int k = 0; k < CS; ++k) cy.v[k] = 0.f;

    // software prefetch of the streaming operands of the next row
    float gx_n = -4.f, gy_n = -4.f, go_n[CS];
#pragma unroll
    for (int k = 0; k < CS; ++k) go_n[k] = 0.f;
    if (col_ok) {
        if (inter) { const float2 v = ldg_pair(gq); gx_n = v.x; gy_n = v.y; }
        else { gx_n = to_acc(ldg(gq)); gy_n = to_acc(ldg(gq + grid.s3)); }
#pragma unroll
        for (int k = 0; k < CS; ++k) go_n[k] = to_acc(ldg(goq + k * go_ch));
    }

    for (int r = 0; r < rows; ++r) {
        const float gx = gx_n, gy = gy_n;
        float go[CS];
#pragma unroll
        for (int k = 0; k < CS; ++k) go[k] = go_n[k];
        gq += grid.s1; goq += gout.s2;
        if (col_ok && r + 1 < rows) {
            if (inter) { const float2 v = ldg_pair(gq); gx_n = v.x; gy_n = v.y; }
            else { gx_n = to_acc(ldg(gq)); gy_n = to_acc(ldg(gq + grid.s3)); }
#pragma unroll
            for (int k = 0; k < CS; ++k) go_n[k] = to_acc(ldg(goq + k * go_ch));
        }
        float gxm, gym;
        const float ix = src_index_grad<kBorder, kAlign>(gx, Wf, Wm1, &gxm);
        const float iy = src_index_grad<kBorder, kAlign>(gy, Hf, Hm1, &gym);
        const bool inside = col_ok && ix >= 0.0f && ix < Wm1 && iy >= 0.0f && iy < Hm1;  // floor in [0, size-2]
        if (__all_sync(0xffffffffu, inside))
            row_body<T, G, CS, kGin, kGgrid, false>(lane, true, live, ix, iy, gxm, gym, go, ip, sH, i_ch, g.H, g.W, gip, gi_ch, ggq, ggrid.s3, cy, queue);
        else
            row_body<T, G, CS, kGin, kGgrid, true>(lane, col_ok, live, ix, iy, gxm, gym, go, ip, sH, i_ch, g.H, g.W, gip, gi_ch, ggq, ggrid.s3, cy, queue);
        if (kGgrid) ggq += ggrid.s1;
    }
    if (kGin && cy.live) {
        const int o_cy = cy.y * sH + cy.x;
#pragma unroll
        for (int k = 0; k < CS; ++k) atomicAdd(gip + (k * gi_ch + o_cy), cy.v[k]);
    }
}

template <typename T, typename G, int CS, bool kBorder, bool kAlign>
void launch_ba(const Problem &pb, dim3 blocks, int n0, cudaStream_t st)
{
    if (pb.want_gin && pb.want_ggrid)
        { bwd_lean_kernel<T, G, CS, kBorder, kAlign, true, true><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, n0); note_launch(); }
    else if (pb.want_gin)
        { bwd_lean_kernel<T, G, CS, kBorder, kAlign, true, false><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, n0); note_launch(); }
    else
        { bwd_lean_kernel<T, G, CS, kBorder, kAlign, false, true><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, n0); note_launch(); }
}

template <typename T, typename G, int CS>
void launch_cs(const Problem &pb, dim3 blocks, int n0, cudaStream_t st)
{
    const bool border = pb.g.padding == PWS_PAD_BORDER, align = pb.g.align != 0;
    if (border && align) launch_ba<T, G, CS, true, true>(pb, blocks, n0, st);
    else if (border) launch_ba<T, G, CS, true, false>(pb, blocks, n0, st);
    else if (align) launch_ba<T, G, CS, false, true>(pb, blocks, n0, st);
    else launch_ba<T, G, CS, false, false>(pb, blocks, n0, st);
}

template <typename T, typename G>
void launch_c(const Problem &pb, dim3 blocks, int n0, cudaStream_t st)
{
    if (pb.g.C == 3) launch_cs<T, G, 3>(pb, blocks, n0, st);
    else launch_cs<T, G, 1>(pb, blocks, n0, st);
}

}  // namespace

bool backward_lean_eligible(const Problem &pb)
{
    const Geometry &g = pb.g;
    if (pb.in_dtype != PWS_F32 && pb.in_dtype != PWS_F16 && pb.in_dtype != PWS_BF16) return false;
    const bool map32 = pb.grid_dtype == PWS_F32;
    if (!map32 && pb.grid_dtype != pb.in_dtype) return false;
    if (g.C != 1 && g.C != 3) return false;
    if (pb.in.s3 != 1 || pb.gout.s3 != 1) return false;
    // the scatter reuses the frame's in-plane offset for grad_input: same pitch required
    if (pb.want_gin && !(pb.gin.s3 == 1 && pb.gin.s2 == pb.in.s2)) return false;
    if (!map_pairs_ok(pb.grid, map32 ? 4 : 2)) return false;
    if (pb.want_ggrid && !map_pairs_ok(pb.ggrid, map32 ? 4 : 2)) return false;
    if ((g.Ho + kTH - 1) / kTH > 65535) return false;
    return true;
}

// Launch frames [n0, n0+nn) of an eligible problem.
void launch_backward_lean(const Problem &pb, int n0, int nn, cudaStream_t st)
{
    const Geometry &g = pb.g;
    for (int z0 = 0; z0 < nn; z0 += 65535) {
        const int nz = nn - z0 < 65535 ? nn - z0 : 65535;
        dim3 blocks((g.Wo + kTW - 1) / kTW, (g.Ho + kTH - 1) / kTH, nz);
        const bool map32 = pb.grid_dtype == PWS_F32;
        if (pb.in_dtype == PWS_F32) launch_c<float, float>(pb, blocks, n0 + z0, st);
        else if (pb.in_dtype == PWS_F16) { if (map32) launch_c<__half, float>(pb, blocks, n0 + z0, st); else launch_c<__half, __half>(pb, blocks, n0 + z0, st); }
        else { if (map32) launch_c<__nv_bfloat16, float>(pb, blocks, n0 + z0, st); else launch_c<__nv_bfloat16, __nv_bfloat16>(pb, blocks, n0 + z0, st); }
    }
}

}  // namespace pws
