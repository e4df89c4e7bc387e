// warp_fwd_tile.cu -- lean direct-gather forward warp for the reference's hot layouts (fallback of warp_fwd_tma.cu).
//
// Call sites: R/main_new.py:106,116 (NCHW frames, planar-stored maps), :197 (NCHW
// frames, interleaved affine_grid maps), :716 (same at native video resolution).
// Host-checked requirements: frame and output W-contiguous and 16-byte row aligned,
// C in {1,3}, f32 / f16 / bf16 frames, an fp32 map or one of the frame's 16-bit type.  Everything else takes the direct
// kernel (warp_fwd.cu).
#include "pws_tile.cuh"

#include <cstdlib>

namespace pws {

namespace {

constexpr int kTW = 64, kTH = 32, kBW = 80, kBH = 40, kThreads = 256, kWarps = 8;
constexpr int kPX = kTW / 32, kPY = kTH / kWarps;

// Layout-specialised direct gather: taps through L1 (no staging, no barrier).  4 pixels per thread, 64x16 tile.
// G: map element type (float, or T for 16-bit frames); map coordinates are upcast to fp32 on load.
template <typename T, typename G, int CS, bool kBorder, bool kAlign>
#ifndef PWS_FWD_MINB
#define PWS_FWD_MINB 5   // 48 registers, 40 warps/SM: measured ~7 % faster than 4 CTAs at 56 registers
#endif
__global__ void __launch_bounds__(kThreads, PWS_FWD_MINB)
fwd_lean_kernel(const View in, const View grid, const View out, const Geometry g)
{
    constexpr int PY = 2;
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int n = blockIdx.z;
    const int w_base = blockIdx.x * kTW + lane, h_base = blockIdx.y * (kWarps * PY) + wrp;
    const G *__restrict__ gp = (const G *)grid.p + (int64_t)n * grid.sN;
    const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
    T *__restrict__ op = (T *)out.p + (int64_t)n * out.sN;
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);
    const bool full = (blockIdx.x + 1) * kTW <= g.Wo && (blockIdx.y + 1) * (kWarps * PY) <= g.Ho;

    float sx[PY][kPX], sy[PY][kPX];
    {
        const bool inter = grid.s3 == 1;
        const G *__restrict__ q = gp + (int64_t)h_base * grid.s1 + (int64_t)w_base * grid.s2;
        const int64_t row = (int64_t)kWarps * grid.s1;
        const int col = 32 * grid.s2;
#pragma unroll
        for (int j = 0; j < PY; ++j)
#pragma unroll
            for (int i = 0; i < kPX; ++i) {
                sx[j][i] = -4.0f; sy[j][i] = -4.0f;
                if (full || (w_base + 32 * i < g.Wo && h_base + kWarps * j < g.Ho)) {
                    const G *__restrict__ a = q + j * row + i * col;
                    if (inter) {
                        const float2 v = ldg_pair(a);
                        sx[j][i] = v.x; sy[j][i] = v.y;
                    } else {
                        sx[j][i] = to_acc(ldg(a));
                        sy[j][i] = to_acc(ldg(a + grid.s3));
                    }
                }
            }
    }
    const int o_row = kWarps * out.s2, o_ch = out.s1, i_ch = in.s1;  // 32-bit in-frame offsets
    const int sH = in.s2;
    T *__restrict__ o0 = op + (int64_t)h_base * out.s2 + w_base;
#pragma unroll
    for (int j = 0; j < PY; ++j)
#pragma unroll
        for (int i = 0; i < kPX; ++i) {
            const bool ok = full || (w_base + 32 * i < g.Wo && h_base + kWarps * j < g.Ho);
            const float ix = src_index<kBorder, kAlign>(sx[j][i], g.W, Wf, Wm1);
            const float iy = src_index<kBorder, kAlign>(sy[j][i], g.H, Hf, Hm1);
            const float x0f = floorf(ix), y0f = floorf(iy);
            const bool inside = x0f >= 0.0f && x0f <= Wm1 - 1.0f && y0f >= 0.0f && y0f <= Hm1 - 1.0f;
            T *__restrict__ o = o0 + (j * o_row + 32 * i);
            if (__all_sync(0xffffffffu, inside && ok)) {
                const float wx1 = fsub(ix, x0f), wx0 = fsub(x0f + 1.0f, ix);
                const float wy1 = fsub(iy, y0f), wy0 = fsub(y0f + 1.0f, iy);
                const float nw = fmul(wx0, wy0), ne = fmul(wx1, wy0), sw = fmul(wx0, wy1), se = fmul(wx1, wy1);
                const T *__restrict__ p0 = ip + ((int)y0f * sH + (int)x0f);
#pragma unroll
                for (int c = 0; c < CS; ++c) {
                    const T *__restrict__ pc = p0 + c * i_ch;
                    const float v0 = to_acc(ldg(pc)), v1 = to_acc(ldg(pc + 1));
                    const float v2 = to_acc(ldg(pc + sH)), v3 = to_acc(ldg(pc + sH + 1));
                    float acc = ffma(v0, nw, 0.f);
                    acc = ffma(v1, ne, acc);
                    acc = ffma(v2, sw, acc);
                    acc = ffma(v3, se, acc);
                    o[c * o_ch] = from_acc<T, float>(acc);
                }
            } else if (ok) {
                Taps<float> t;
                make_taps(ix, iy, g.H, g.W, t);
                const T *__restrict__ p0 = ip + (t.y0 * sH + t.x0);
#pragma unroll
                for (int c = 0; c < CS; ++c) {
                    const T *__restrict__ pc = p0 + c * i_ch;
                    float acc = 0.f;
                    if (t.mask & 1u) acc = ffma(to_acc(ldg(pc)), t.nw, acc);
                    if (t.mask & 2u) acc = ffma(to_acc(ldg(pc + 1)), t.ne, acc);
                    if (t.mask & 4u) acc = ffma(to_acc(ldg(pc + sH)), t.sw, acc);
                    if (t.mask & 8u) acc = ffma(to_acc(ldg(pc + sH + 1)), t.se, acc);
                    o[c * o_ch] = from_acc<T, float>(acc);
                }
            }
        }
}

template <typename T, typename G, int CS>
void launch_cs(const Problem &pb, cudaStream_t st)
{
    const Geometry &g = pb.g;
    const bool border = g.padding == PWS_PAD_BORDER, align = g.align != 0;
    {
        dim3 lb((g.Wo + kTW - 1) / kTW, (g.Ho + 15) / 16, g.N);
        if (border && align) { fwd_lean_kernel<T, G, CS, true, true><<<lb, kThreads, 0, st>>>(pb.in, pb.grid, pb.out, g); note_launch(); }
        else if (border) { fwd_lean_kernel<T, G, CS, true, false><<<lb, kThreads, 0, st>>>(pb.in, pb.grid, pb.out, g); note_launch(); }
        else if (align) { fwd_lean_kernel<T, G, CS, false, true><<<lb, kThreads, 0, st>>>(pb.in, pb.grid, pb.out, g); note_launch(); }
        else { fwd_lean_kernel<T, G, CS, false, false><<<lb, kThreads, 0, st>>>(pb.in, pb.grid, pb.out, g); note_launch(); }
    }
}

template <typename T, typename G>
bool launch_t(const Problem &pb, cudaStream_t st)
{
    if (!rows_vectorizable(pb.in, 16 / (int)sizeof(T), pb.g.W)) return false;
    if (pb.g.C == 3) { launch_cs<T, G, 3>(pb, st); return true; }
    if (pb.g.C == 1) { launch_cs<T, G, 1>(pb, st); return true; }
    return false;
}

}  // namespace

// Returns true when the lean kernel took the call.
bool launch_forward_tile(const Problem &pb, cudaStream_t st)
{
    const Geometry &g = pb.g;
    if (pb.in.s3 != 1 || pb.out.s3 != 1) return false;
    if (g.N > 65535 || (g.Ho + kTH - 1) / kTH > 65535) return false;
    const bool map32 = pb.grid_dtype == PWS_F32;
    if (!map32 && pb.grid_dtype != pb.in_dtype) return false;
    if (!map_pairs_ok(pb.grid, map32 ? 4 : 2)) return false;
    if (pb.in_dtype == PWS_F32) return map32 && launch_t<float, float>(pb, st);
    if (pb.in_dtype == PWS_F16) return map32 ? launch_t<__half, float>(pb, st) : launch_t<__half, __half>(pb, st);
    if (pb.in_dtype == PWS_BF16) return map32 ? launch_t<__nv_bfloat16, float>(pb, st) : launch_t<__nv_bfloat16, __nv_bfloat16>(pb, st);
    return false;
}

}  // namespace pws
