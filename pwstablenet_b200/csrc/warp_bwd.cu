// warp_bwd.cu -- backward pixel-wise warp: grad to the frame (scatter) and to the map.
//
// Replaces launch_grid_sampler_2d_backward_kernel ($TORCH/include/ATen/native/cuda/GridSampler.h:16-24),
// reached from loss_g.backward() at R/main_new.py:214 for the warps at :106,116,197.
//
// ATen issues 4*C global float atomics per output pixel (59 REDG in its sm_100
// SASS, no SHFL/LDS: SURVEY.md 2.2).  Here a warp owns a 32-pixel-wide strip and
// marches down kRows output rows:
//   * horizontally, lane i's east taps (x0+1, y0 / y0+1) are the west taps of lane
//     i+1 whenever the map advances one source pixel per output pixel -- lane i+1
//     takes them over with two shuffles per channel instead of two atomics;
//   * vertically, the south taps of row r are the north taps of row r+1 when the
//     map advances one source row -- they are carried in registers to the next
//     iteration instead of being written.
// What is left is ~1 RED per source pixel and channel, lanes hitting consecutive
// addresses (one 128-byte L2 atomic request per warp instruction), plus the
// strip-edge remainders.  Irregular maps simply match less often and fall back
// towards ATen's 4 atomics per pixel; correctness never depends on a match.
// Shared-memory float atomics are NOT used on this path: on sm_100a
// atomicAdd(float*) on shared memory compiles to an ATOMS.CAST.SPIN loop
// (DESIGN.md "backward"), slower than the L2's native RED.ADD.F32.
//
// grad_input is zero-filled by the library, one chunk of frames at a time, right
// before the kernel that scatters into that chunk: the zeroed lines are still
// dirty in the 126 MB L2 when the REDs arrive, so grad_input costs one DRAM write
// instead of write + read + write.
#include "pws_common.cuh"

#include <cstdlib>

namespace pws {

namespace {

constexpr int kRows = 16;           // output rows a warp marches over
constexpr int kWarpsX = 2, kWarpsY = 4;
constexpr int kThreads = 32 * kWarpsX * kWarpsY;
constexpr int kTileW = 32 * kWarpsX, kTileH = kRows * kWarpsY;

template <typename T> __device__ __forceinline__ void red_add(T *p, T v) { atomicAdd(p, v); }

// grad_grid of one pixel over all C channels in one pass, for maps too narrow to park partial sums between channel chunks:
// the fma chain of bwd_march_kernel, channel after channel, rounded to G once
template <typename T, typename G, typename A>
__device__ __forceinline__ void ggrid_all_channels(const T *__restrict__ gop, const T *__restrict__ ip, G *__restrict__ ggp,
                                                   const View &gout, const View &in, const View &ggrid, const Geometry &g,
                                                   const Taps<A> &t, const A gxm, const A gym, const int h, const int w)
{
    const A x0f = (A)t.x0, y0f = (A)t.y0, x1f = (A)(t.x0 + 1), y1f = (A)(t.y0 + 1);
    const A dn = fsub(y1f, t.iy), ds = fsub(t.iy, y0f), dw = fsub(x1f, t.ix), de = fsub(t.ix, x0f);
    const int o_nw = t.y0 * in.s2 + t.x0 * in.s3;
    const T *__restrict__ goc = gop + h * gout.s2 + w * gout.s3;
    A gix = (A)0, giy = (A)0;
    for (int c = 0; c < g.C; ++c) {
        const A go = to_acc(ldg(goc + c * gout.s1));
        const T *__restrict__ pc = ip + c * in.s1;
        A v0 = (A)0, v1 = (A)0, v2 = (A)0, v3 = (A)0;
        if (t.mask & 1u) v0 = to_acc(ldg(pc + o_nw));
        if (t.mask & 2u) v1 = to_acc(ldg(pc + o_nw + in.s3));
        if (t.mask & 4u) v2 = to_acc(ldg(pc + o_nw + in.s2));
        if (t.mask & 8u) v3 = to_acc(ldg(pc + o_nw + in.s2 + in.s3));
        if (t.mask & 1u) { gix = ffma(-fmul(v0, dn), go, gix); giy = ffma(-fmul(v0, dw), go, giy); }
        if (t.mask & 2u) { gix = ffma(fmul(v1, dn), go, gix);  giy = ffma(-fmul(v1, de), go, giy); }
        if (t.mask & 4u) { gix = ffma(-fmul(v2, ds), go, gix); giy = ffma(fmul(v2, dw), go, giy); }
        if (t.mask & 8u) { gix = ffma(fmul(v3, ds), go, gix);  giy = ffma(fmul(v3, de), go, giy); }
    }
    const int off = h * ggrid.s1 + w * ggrid.s2;
    ggp[off] = from_acc<G, A>(fmul(gxm, gix));
    ggp[off + ggrid.s3] = from_acc<G, A>(fmul(gym, giy));
}

// T: element type of the frame and of grad_output; G: of the map and of grad_grid (T, or float for 16-bit frames).
// grad_input is written in the accumulation type (fp32 for 16-bit frames: the caller rounds the sums once).
template <typename T, typename G, int CS, bool kGin, bool kGgrid>
__global__ void __launch_bounds__(kThreads)
bwd_march_kernel(const View gout, const View in, const View grid, const View gin, const View ggrid,
                 const Geometry g, const int tiles_x, const int tiles_y, const int n_begin)
{
    using A = typename Acc<T>::type;
    // grad_grid can hold the raw partial sums between channel chunks only when it is at least as wide as the accumulator;
    // a 16-bit grad_grid would round them, so those maps sum every channel in registers during the first chunk instead
    constexpr bool kPark = sizeof(G) >= sizeof(A);
    const int tile = blockIdx.x;
    const int tx = tile % tiles_x;
    const int rest = tile / tiles_x;
    const int ty = rest % tiles_y;
    const int n = n_begin + rest / tiles_y;
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int w = tx * kTileW + (wrp % kWarpsX) * 32 + lane;
    const int h0 = ty * kTileH + (wrp / kWarpsX) * kRows;
    if (h0 >= g.Ho) return;  // warp-uniform
    const bool col_ok = w < g.Wo;
    const bool align = g.align != 0;

    const T *__restrict__ gop = (const T *)gout.p + (int64_t)n * gout.sN;
    const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
    const G *__restrict__ gp = (const G *)grid.p + (int64_t)n * grid.sN;
    A *__restrict__ gip = kGin ? (A *)gin.p + (int64_t)n * gin.sN : nullptr;
    G *__restrict__ ggp = kGgrid ? (G *)ggrid.p + (int64_t)n * ggrid.sN : nullptr;

    const int rows = min(kRows, g.Ho - h0);

    for (int c0 = 0; c0 < g.C; c0 += CS) {
        // vertical carry: the south-west totals of the previous row
        int carry_x = 0, carry_y = 0;
        bool carry_live = false;  // target in bounds and worth flushing
        A carry_v[CS];
#pragma unroll
        for (int k = 0; k < CS; ++k) carry_v[k] = (A)0;

        // software prefetch of the streaming operands of the next row
        A gx_n = (A)0, gy_n = (A)0, go_n[CS];
#pragma unroll
        for (int k = 0; k < CS; ++k) go_n[k] = (A)0;
        if (col_ok) {
            const int off = h0 * grid.s1 + w * grid.s2;
            gx_n = to_acc(ldg(gp + off));
            gy_n = to_acc(ldg(gp + off + grid.s3));
#pragma unroll
            for (int k = 0; k < CS; ++k) go_n[k] = to_acc(ldg(gop + (c0 + k) * gout.s1 + h0 * gout.s2 + w * gout.s3));
        }

        for (int r = 0; r < rows; ++r) {
            const int h = h0 + r;
            const A gx = gx_n, gy = gy_n;
            A go[CS];
#pragma unroll
            for (int k = 0; k < CS; ++k) go[k] = go_n[k];
            if (col_ok && r + 1 < rows) {
                const int off = (h + 1) * grid.s1 + w * grid.s2;
                gx_n = to_acc(ldg(gp + off));
                gy_n = to_acc(ldg(gp + off + grid.s3));
#pragma unroll
                for (int k = 0; k < CS; ++k)
                    go_n[k] = to_acc(ldg(gop + (c0 + k) * gout.s1 + (h + 1) * gout.s2 + w * gout.s3));
            }

            A gxm, gym;
            Taps<A> t;
            {
                const A ix = source_index_set_grad(gx, g.W, g.padding, align, &gxm);
                const A iy = source_index_set_grad(gy, g.H, g.padding, align, &gym);
                make_taps(ix, iy, g.H, g.W, t);
            }
            if (!col_ok) t.mask = 0u;

            if (kPark && kGgrid && col_ok) {
                const A x0f = (A)t.x0, y0f = (A)t.y0, x1f = (A)(t.x0 + 1), y1f = (A)(t.y0 + 1);
                const A dn = fsub(y1f, t.iy), ds = fsub(t.iy, y0f), dw = fsub(x1f, t.ix), de = fsub(t.ix, x0f);
                const int o_nw = t.y0 * in.s2 + t.x0 * in.s3;
                const int off = h * ggrid.s1 + w * ggrid.s2;
                // channel chunks after the first continue the fma chain from the raw partial sums the
                // previous chunk parked in grad_grid, so the result equals one pass over all channels
                A gix = (A)0, giy = (A)0;
                if (c0 > 0) { gix = to_acc(ggp[off]); giy = to_acc(ggp[off + ggrid.s3]); }
#pragma unroll
                for (int k = 0; k < CS; ++k) {
                    const T *__restrict__ pc = ip + (c0 + k) * in.s1;
                    A v0 = (A)0, v1 = (A)0, v2 = (A)0, v3 = (A)0;
                    if (t.mask & 1u) v0 = to_acc(ldg(pc + o_nw));
                    if (t.mask & 2u) v1 = to_acc(ldg(pc + o_nw + in.s3));
                    if (t.mask & 4u) v2 = to_acc(ldg(pc + o_nw + in.s2));
                    if (t.mask & 8u) v3 = to_acc(ldg(pc + o_nw + in.s2 + in.s3));
                    // ATen's statement order; t = v*d rounded, then one fma with gOut
                    if (t.mask & 1u) { gix = ffma(-fmul(v0, dn), go[k], gix); giy = ffma(-fmul(v0, dw), go[k], giy); }
                    if (t.mask & 2u) { gix = ffma(fmul(v1, dn), go[k], gix);  giy = ffma(-fmul(v1, de), go[k], giy); }
                    if (t.mask & 4u) { gix = ffma(-fmul(v2, ds), go[k], gix); giy = ffma(fmul(v2, dw), go[k], giy); }
                    if (t.mask & 8u) { gix = ffma(fmul(v3, ds), go[k], gix);  giy = ffma(fmul(v3, de), go[k], giy); }
                }
                if (c0 + CS >= g.C) { gix = fmul(gxm, gix); giy = fmul(gym, giy); }
                ggp[off] = from_acc<G, A>(gix);
                ggp[off + ggrid.s3] = from_acc<G, A>(giy);
            }
            if constexpr (!kPark) {
                if (kGgrid && col_ok && c0 == 0) ggrid_all_channels<T, G>(gop, ip, ggp, gout, in, ggrid, g, t, gxm, gym, h, w);
            }

            if (kGin) {
                // who is next to me, and do our taps chain?
                const unsigned live = __ballot_sync(0xffffffffu, col_ok);
                const int px0 = __shfl_up_sync(0xffffffffu, t.x0, 1), py0 = __shfl_up_sync(0xffffffffu, t.y0, 1);
                const int nx0 = __shfl_down_sync(0xffffffffu, t.x0, 1), ny0 = __shfl_down_sync(0xffffffffu, t.y0, 1);
                const bool take = col_ok && lane > 0 && ((live >> (lane - 1)) & 1u) && px0 + 1 == t.x0 && py0 == t.y0;
                const bool given = col_ok && lane < 31 && ((live >> (lane + 1)) & 1u) && nx0 == t.x0 + 1 && ny0 == t.y0;
                const bool chain = carry_live && carry_x == t.x0 && carry_y == t.y0;
                const int o_nw = t.y0 * gin.s2 + t.x0 * gin.s3;
                const int o_carry = carry_y * gin.s2 + carry_x * gin.s3;
#pragma unroll
                for (int k = 0; k < CS; ++k) {
                    A *__restrict__ pc = gip + (c0 + k) * gin.s1;
                    A top = fmul(t.nw, go[k]), bot = fmul(t.sw, go[k]);
                    const A etop = fmul(t.ne, go[k]), ebot = fmul(t.se, go[k]);
                    const A ptop = __shfl_up_sync(0xffffffffu, etop, 1), pbot = __shfl_up_sync(0xffffffffu, ebot, 1);
                    if (take) { top += ptop; bot += pbot; }
                    if (!given) {
                        if (t.mask & 2u) red_add(pc + o_nw + gin.s3, etop);
                        if (t.mask & 8u) red_add(pc + o_nw + gin.s2 + gin.s3, ebot);
                    }
                    if (chain) top += carry_v[k];
                    else if (carry_live) red_add(pc + o_carry, carry_v[k]);
                    if (t.mask & 1u) red_add(pc + o_nw, top);
                    carry_v[k] = bot;
                }
                carry_x = t.x0; carry_y = t.y0 + 1;
                carry_live = (t.mask & 4u) != 0u;
            }
        }
        if (kGin && carry_live) {
            const int o_carry = carry_y * gin.s2 + carry_x * gin.s3;
#pragma unroll
            for (int k = 0; k < CS; ++k) red_add(gip + (c0 + k) * gin.s1 + o_carry, carry_v[k]);
        }
    }
}

template <typename T, typename G, int CS>
void launch_cs(const Problem &pb, unsigned blocks, int tiles_x, int tiles_y, int n_begin, cudaStream_t st)
{
    if (pb.want_gin && pb.want_ggrid)
        { bwd_march_kernel<T, G, CS, true, true><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, tiles_x, tiles_y, n_begin); note_launch(); }
    else if (pb.want_gin)
        { bwd_march_kernel<T, G, CS, true, false><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, tiles_x, tiles_y, n_begin); note_launch(); }
    else
        { bwd_march_kernel<T, G, CS, false, true><<<blocks, kThreads, 0, st>>>(pb.gout, pb.in, pb.grid, pb.gin, pb.ggrid, pb.g, tiles_x, tiles_y, n_begin); note_launch(); }
}

}  // namespace
bool backward_lean_eligible(const Problem &pb);                                  // warp_bwd_lean.cu
void launch_backward_lean(const Problem &pb, int n0, int nn, cudaStream_t st);   // warp_bwd_lean.cu
struct BwdTmaPlan;                                                               // warp_bwd_tma.cu
BwdTmaPlan *backward_tma_plan(const Problem &pb);
void backward_tma_free(BwdTmaPlan *pl);
bool launch_backward_tma(const BwdTmaPlan *pl, const Problem &pb, int n0, int nn, cudaStream_t st);
int backward_tma_max_frames();
namespace {

bool force_generic()
{
#ifdef PWS_DEV_HOOKS
    static const bool v = [] { const char *e = std::getenv("PWS_FORCE_DIRECT"); return e && e[0] == '1'; }();
    return v;
#else
    return false;
#endif
}

int64_t chunk_bytes()
{
    // grad_input bytes zero-filled ahead of each scatter launch; must stay well inside L2
    // (measured: while the kernel is issue-bound one launch beats L2-sized chunks)
    return (int64_t)4096 << 20;
}

// The whole backward through the persistent TMA kernel, backward_tma_max_frames() frames per launch; the kernel
// zero-fills grad_input itself, a few bands ahead of its scatter: no memset pass.  false: the kernel cannot take the
// problem or refused a launch (stream capture, a context too small for the cooperative launch); the caller's fallback
// then redoes every frame.
bool backward_tma(const Problem &pb, cudaStream_t st)
{
    BwdTmaPlan *plan = backward_tma_plan(pb);
    if (!plan) return false;
    const int step = backward_tma_max_frames();
    bool ok = true;
    for (int n0 = 0; ok && n0 < pb.g.N; n0 += step) ok = launch_backward_tma(plan, pb, n0, pb.g.N - n0 < step ? pb.g.N - n0 : step, st);
    backward_tma_free(plan);
    return ok;
}

// f32 / f64 problems (TMA, lean or march kernel), and the march kernel for 16-bit frames (T 16-bit; grad_input is then the
// fp32 accumulation buffer, so the zero-fill is sized by the accumulator type, not by T)
template <typename T, typename G>
int launch_typed(const Problem &pb, cudaStream_t st)
{
    const Geometry &g = pb.g;
    const int tiles_x = (g.Wo + kTileW - 1) / kTileW, tiles_y = (g.Ho + kTileH - 1) / kTileH;
    const int64_t gin_elem = (int64_t)sizeof(typename Acc<T>::type);
    const int64_t frame_bytes = (int64_t)g.C * g.H * g.W * gin_elem;
    int per_chunk = g.N;
    if (pb.want_gin) {
        per_chunk = (int)(chunk_bytes() / (frame_bytes > 0 ? frame_bytes : 1));
        if (per_chunk < 1) per_chunk = 1;
        if (per_chunk > g.N) per_chunk = g.N;
    }
    const bool lean = sizeof(T) == 4 && !force_generic() && backward_lean_eligible(pb);
    if (sizeof(T) == 4 && !force_generic() && !(lean && small_problem(pb)) && backward_tma(pb, st)) return PWS_OK;
    // 16-bit frames chunk at most 2 channels: their CS = 4 instantiation spills (128 registers)
    constexpr int kCs4 = sizeof(T) == 2 ? 2 : 4;
    const int cs = (g.C == 3) ? 3 : (g.C % kCs4 == 0) ? kCs4 : (g.C % 2 == 0) ? 2 : 1;
    for (int n0 = 0; n0 < g.N; n0 += per_chunk) {
        const int nn = (g.N - n0 < per_chunk) ? g.N - n0 : per_chunk;
        if (pb.want_gin) {
            cudaError_t e = cudaMemsetAsync((char *)pb.gin.p + (int64_t)n0 * pb.gin.sN * gin_elem, 0,
                                            (size_t)(frame_bytes * nn), st);
            if (e != cudaSuccess) { set_error("backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
        }
        note_kernel(lean ? "bwd_lean" : sizeof(T) == 2 ? "bwd_march_16" : "bwd_march");
        if (lean) { launch_backward_lean(pb, n0, nn, st); continue; }
        const int64_t tiles = (int64_t)tiles_x * tiles_y * nn;
        if (tiles == 0) continue;
        if (tiles > INT_MAX) { set_error("backward: too many tiles"); return PWS_EUNSUPPORTED; }
        switch (cs) {
            case 3: launch_cs<T, G, 3>(pb, (unsigned)tiles, tiles_x, tiles_y, n0, st); break;
            case 4: launch_cs<T, G, kCs4>(pb, (unsigned)tiles, tiles_x, tiles_y, n0, st); break;
            case 2: launch_cs<T, G, 2>(pb, (unsigned)tiles, tiles_x, tiles_y, n0, st); break;
            default: launch_cs<T, G, 1>(pb, (unsigned)tiles, tiles_x, tiles_y, n0, st); break;
        }
    }
    return PWS_OK;
}

// 16-bit frames and grad_output with an fp32 map (BASELINE config 5) or a map of the frame's type: fp32 arithmetic, grad_grid
// rounded to the map's type once, and an fp32 grad_input ACCUMULATION buffer (capi.cu requires it), which the caller rounds
// to the frame type once -- summing a pixel's contributions in bf16 would round after every atomic.
int launch_16bit(const Problem &pb, cudaStream_t st)
{
    // above the small-problem threshold: the persistent TMA kernel with 16-bit grad_output tiles and frame boxes (RGB, fp32
    // maps only)
    if (!force_generic() && !small_problem(pb) && backward_tma(pb, st)) return PWS_OK;
    if (!backward_lean_eligible(pb)) {
        // any C, strides, channels-last or cropped frames: the marching kernel
        const bool map32 = pb.grid_dtype == PWS_F32;
        if (pb.in_dtype == PWS_F16) return map32 ? launch_typed<__half, float>(pb, st) : launch_typed<__half, __half>(pb, st);
        return map32 ? launch_typed<__nv_bfloat16, float>(pb, st) : launch_typed<__nv_bfloat16, __nv_bfloat16>(pb, st);
    }
    const Geometry &g = pb.g;
    if (pb.want_gin) {
        cudaError_t e = cudaMemsetAsync(pb.gin.p, 0, (size_t)g.N * pb.gin.sN * sizeof(float), st);
        if (e != cudaSuccess) { set_error("backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
    }
    note_kernel("bwd_lean_16");
    launch_backward_lean(pb, 0, g.N, st);
    return PWS_OK;
}

}  // namespace

int launch_backward(const Problem &pb, cudaStream_t st)
{
    if (!pb.want_gin && !pb.want_ggrid) return PWS_OK;
    if (pb.in_dtype != pb.grid_dtype && !(pb.grid_dtype == PWS_F32 && (pb.in_dtype == PWS_F16 || pb.in_dtype == PWS_BF16))) {
        set_error("backward: frame and map dtypes must match, or 16-bit frames with an fp32 map (got %d, %d)", pb.in_dtype, pb.grid_dtype);
        return PWS_EUNSUPPORTED;
    }
    if (pb.in_dtype == PWS_F16 || pb.in_dtype == PWS_BF16) return launch_16bit(pb, st);
    if (pb.in_dtype == PWS_F32) return launch_typed<float, float>(pb, st);
    if (pb.in_dtype == PWS_F64) return launch_typed<double, double>(pb, st);
    set_error("backward: unsupported dtype %d", pb.in_dtype);
    return PWS_EUNSUPPORTED;
}

}  // namespace pws
