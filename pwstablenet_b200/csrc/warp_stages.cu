// warp_stages.cu -- K maps applied to the SAME frame in one launch, pre / post scale folded in, forward and backward.
//
// R/main_new.py:103-110 (and :112-119 for the second clip): the three cascade stages of netG each emit a complete map,
// and every map samples the SAME unstable frame:
//     for nl in range(3):  fake = grid_sample((rgb + 1) * 127.5, grid1[nl]) / 127.5 - 1
// The reference runs that as 3 elementwise passes + 3 sampler launches + 6 more elementwise passes per clip, each one a
// launch-bound kernel on a 12.6 MB working set.  Here one launch reads the raw frame, applies (x + a) * b to the taps,
// samples with every map and writes acc * m + e for each: the scaled frame and the unscaled samples never exist.  The
// maps of the cascade are refinements of each other, so the taps of stage k + 1 are the taps of stage k for most pixels
// and stay in registers (the frame is read once, not K times).
// Backward (autograd of the above, R/main_new.py:214): grad_grid of every stage from the stage's grad_output, with the
// chain rule through the post scale (grad * m, as autograd computes it for `x / 127.5`: a multiplication by the rounded
// reciprocal) and the taps pre-scaled as in the forward; optional grad_input (direct REDs: the training sites never ask).
// Arithmetic is statement for statement that of the unfused torch pipeline: (x + a) * b rounded per tap, ATen's sampler
// order (pws_common.cuh), `acc * m` then `+ e` -- results are bit-identical to the reference's sequence of torch calls.
// 16-bit frames (T = __half / __nv_bfloat16, maps G = float or T): that sequence on a half-precision tensor computes every
// elementwise op in fp32 and rounds it to T, and the sampler rounds once; rnd<T> reproduces each of those roundings and is
// the identity for T = float.  Taps and map values are upcast on load, the rest is the fp32 arithmetic; grad_grid is
// rounded once to G, grad_input stays an fp32 accumulation buffer.
#include "pws_common.cuh"

namespace pws {

namespace {

constexpr int kTileW = 64, kTileH = 16, kThreads = 256;

// one elementwise torch op on a T tensor: fp32 result rounded to T (read back as fp32 for the next op)
template <typename T> __device__ __forceinline__ float rnd(float v) { return to_acc(from_acc<T, float>(v)); }

template <bool kBorder, bool kAlign>
__device__ __forceinline__ float src_index_b(float coord, float size_f, float size_m1_f, float *gm)
{
    const float t = __fadd_rn(coord, 1.0f);
    float c = kAlign ? __fmul_rn(__fmul_rn(t, 0.5f), size_m1_f) : __fmul_rn(__fmaf_rn(t, size_f, -1.0f), 0.5f);
    float m = kAlign ? size_m1_f * 0.5f : size_f * 0.5f;
    if (kBorder) {
        if (c <= 0.0f) { c = 0.0f; m = 0.0f; }
        else if (c >= size_m1_f) { c = size_m1_f; m = 0.0f; }
    }
    if (!(c <= 2147483648.0f && c >= -2147483648.0f)) c = -100.0f;
    *gm = m;
    return c;
}

// forward flavour: border padding clips with min / max, which maps a NaN coordinate to 0 (ATen's clip_coordinates),
// where the backward's comparison chain above leaves it NaN (-> the -100 guard)
template <bool kBorder, bool kAlign>
__device__ __forceinline__ float src_index_f(float coord, float size_f, float size_m1_f)
{
    const float t = __fadd_rn(coord, 1.0f);
    float c = kAlign ? __fmul_rn(__fmul_rn(t, 0.5f), size_m1_f) : __fmul_rn(__fmaf_rn(t, size_f, -1.0f), 0.5f);
    if (kBorder) c = fminf(size_m1_f, fmaxf(c, 0.0f));
    if (!(c <= 2147483648.0f && c >= -2147483648.0f)) c = -100.0f;
    return c;
}

// the four taps of every channel of one source pixel position, pre-scaled; reloaded only when the position changes
template <int CS>
struct TapCache {
    int x0, y0;
    float v[CS][4];
};

template <typename T, int CS>
__device__ __forceinline__ void load_taps(TapCache<CS> &tc, const T *__restrict__ ip, const View &in, const Taps<float> &t,
                                          const StageScale &sc)
{
    if (tc.x0 == t.x0 && tc.y0 == t.y0) return;
    tc.x0 = t.x0; tc.y0 = t.y0;
    const int o_nw = t.y0 * in.s2 + t.x0 * in.s3;
#pragma unroll
    for (int c = 0; c < CS; ++c) {
        const T *__restrict__ pc = ip + c * in.s1 + o_nw;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
        if (t.mask & 1u) v0 = to_acc(ldg(pc));
        if (t.mask & 2u) v1 = to_acc(ldg(pc + in.s3));
        if (t.mask & 4u) v2 = to_acc(ldg(pc + in.s2));
        if (t.mask & 8u) v3 = to_acc(ldg(pc + in.s2 + in.s3));
        if (sc.has_pre) {   // (x + a) * b, elementwise as the reference does before sampling: two ops, two roundings to T
            v0 = rnd<T>(__fmul_rn(rnd<T>(__fadd_rn(v0, sc.pre_add)), sc.pre_mul));
            v1 = rnd<T>(__fmul_rn(rnd<T>(__fadd_rn(v1, sc.pre_add)), sc.pre_mul));
            v2 = rnd<T>(__fmul_rn(rnd<T>(__fadd_rn(v2, sc.pre_add)), sc.pre_mul));
            v3 = rnd<T>(__fmul_rn(rnd<T>(__fadd_rn(v3, sc.pre_add)), sc.pre_mul));
        }
        tc.v[c][0] = v0; tc.v[c][1] = v1; tc.v[c][2] = v2; tc.v[c][3] = v3;
    }
}

template <typename T, typename G, int CS, bool kBorder, bool kAlign>
__global__ void __launch_bounds__(kThreads)
stages_fwd_kernel(const View in, const StageViews sv, const int K, const Geometry g, const StageScale sc)
{
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, n = blockIdx.z;
    const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
            if (!(w < g.Wo && h < g.Ho)) continue;
            TapCache<CS> tc;
            tc.x0 = INT_MIN; tc.y0 = INT_MIN;
            for (int k = 0; k < K; ++k) {
                const View &mv = sv.map[k];
                const G *mp = (const G *)mv.p + (int64_t)n * mv.sN + h * mv.s1 + w * mv.s2;
                const float ix = src_index_f<kBorder, kAlign>(to_acc(ldg(mp)), Wf, Wm1);
                const float iy = src_index_f<kBorder, kAlign>(to_acc(ldg(mp + mv.s3)), Hf, Hm1);
                Taps<float> t;
                make_taps(ix, iy, g.H, g.W, t);
                // the cache key is the tap position; the mask is a function of it
                load_taps<T, CS>(tc, ip, in, t, sc);
                const View &ov = sv.io[k];
                T *op = (T *)ov.p + (int64_t)n * ov.sN + h * ov.s2 + w * ov.s3;
#pragma unroll
                for (int c = 0; c < CS; ++c) {
                    float acc = 0.f;
                    if (t.mask & 1u) acc = ffma(tc.v[c][0], t.nw, acc);
                    if (t.mask & 2u) acc = ffma(tc.v[c][1], t.ne, acc);
                    if (t.mask & 4u) acc = ffma(tc.v[c][2], t.sw, acc);
                    if (t.mask & 8u) acc = ffma(tc.v[c][3], t.se, acc);
                    acc = rnd<T>(acc);   // the sampler's output tensor
                    if (sc.has_post) acc = __fadd_rn(rnd<T>(__fmul_rn(acc, sc.post_mul)), sc.post_add);
                    op[c * ov.s1] = from_acc<T, float>(acc);
                }
            }
        }
}

template <typename T, typename G, int CS, bool kBorder, bool kAlign, bool kGin>
__global__ void __launch_bounds__(kThreads)
stages_bwd_kernel(const View in, const StageViews sv, const int K, const View gin, const Geometry g, const StageScale sc)
{
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, n = blockIdx.z;
    const T *__restrict__ ip = (const T *)in.p + (int64_t)n * in.sN;
    float *__restrict__ gip = kGin ? (float *)gin.p + (int64_t)n * gin.sN : nullptr;
    const float Wf = (float)g.W, Hf = (float)g.H, Wm1 = (float)(g.W - 1), Hm1 = (float)(g.H - 1);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
            if (!(w < g.Wo && h < g.Ho)) continue;
            TapCache<CS> tc;
            tc.x0 = INT_MIN; tc.y0 = INT_MIN;
            for (int k = 0; k < K; ++k) {
                const View &mv = sv.map[k];
                const G *mp = (const G *)mv.p + (int64_t)n * mv.sN + h * mv.s1 + w * mv.s2;
                float gxm, gym;
                const float ix = src_index_b<kBorder, kAlign>(to_acc(ldg(mp)), Wf, Wm1, &gxm);
                const float iy = src_index_b<kBorder, kAlign>(to_acc(ldg(mp + mv.s3)), Hf, Hm1, &gym);
                Taps<float> t;
                make_taps(ix, iy, g.H, g.W, t);
                load_taps<T, CS>(tc, ip, in, t, sc);
                const float x0f = (float)t.x0, y0f = (float)t.y0;
                const float dw = fsub(x0f + 1.0f, ix), de = fsub(ix, x0f), dn = fsub(y0f + 1.0f, iy), ds = fsub(iy, y0f);
                const View &ov = sv.io[k];
                const T *gop = (const T *)ov.p + (int64_t)n * ov.sN + h * ov.s2 + w * ov.s3;
                float gix = 0.f, giy = 0.f;
#pragma unroll
                for (int c = 0; c < CS; ++c) {
                    float go = to_acc(ldg(gop + c * ov.s1));
                    if (sc.has_post) go = rnd<T>(__fmul_rn(go, sc.post_mul));   // autograd of `x / d`: grad * (1/d), a T tensor
                    const float v0 = tc.v[c][0], v1 = tc.v[c][1], v2 = tc.v[c][2], v3 = tc.v[c][3];
                    // ATen's statement order: t = v*d rounded, then one fma with gOut
                    if (t.mask & 1u) { gix = ffma(-fmul(v0, dn), go, gix); giy = ffma(-fmul(v0, dw), go, giy); }
                    if (t.mask & 2u) { gix = ffma(fmul(v1, dn), go, gix);  giy = ffma(-fmul(v1, de), go, giy); }
                    if (t.mask & 4u) { gix = ffma(-fmul(v2, ds), go, gix); giy = ffma(fmul(v2, dw), go, giy); }
                    if (t.mask & 8u) { gix = ffma(fmul(v3, ds), go, gix);  giy = ffma(fmul(v3, de), go, giy); }
                    if (kGin) {
                        // d out / d frame = w_tap, through the pre scale (x + a) * b: times b
                        const float gs = sc.has_pre ? __fmul_rn(go, sc.pre_mul) : go;
                        float *pc = gip + c * gin.s1 + t.y0 * gin.s2 + t.x0;
                        if (t.mask & 1u) atomicAdd(pc, fmul(t.nw, gs));
                        if (t.mask & 2u) atomicAdd(pc + 1, fmul(t.ne, gs));
                        if (t.mask & 4u) atomicAdd(pc + gin.s2, fmul(t.sw, gs));
                        if (t.mask & 8u) atomicAdd(pc + gin.s2 + 1, fmul(t.se, gs));
                    }
                }
                const View &gv = sv.gg[k];
                if (gv.p) {
                    G *ggp = (G *)gv.p + (int64_t)n * gv.sN + h * gv.s1 + w * gv.s2;
                    ggp[0] = from_acc<G, float>(fmul(gxm, gix));
                    ggp[gv.s3] = from_acc<G, float>(fmul(gym, giy));
                }
            }
        }
}

template <typename T, typename G>
void stages_forward_typed(const View &in, const StageViews &sv, int K, const Geometry &g, const StageScale &sc, cudaStream_t st)
{
    dim3 blocks((g.Wo + kTileW - 1) / kTileW, (g.Ho + kTileH - 1) / kTileH, g.N);
    const bool border = g.padding == PWS_PAD_BORDER, align = g.align != 0;
#define PWS_F(CS) do { \
        if (border && align) stages_fwd_kernel<T, G, CS, true, true><<<blocks, kThreads, 0, st>>>(in, sv, K, g, sc); \
        else if (border) stages_fwd_kernel<T, G, CS, true, false><<<blocks, kThreads, 0, st>>>(in, sv, K, g, sc); \
        else if (align) stages_fwd_kernel<T, G, CS, false, true><<<blocks, kThreads, 0, st>>>(in, sv, K, g, sc); \
        else stages_fwd_kernel<T, G, CS, false, false><<<blocks, kThreads, 0, st>>>(in, sv, K, g, sc); } while (0)
    if (g.C == 3) PWS_F(3); else PWS_F(1);
#undef PWS_F
}

template <typename T, typename G>
void stages_backward_typed(const View &in, const StageViews &sv, int K, const View &gin, bool want_gin, const Geometry &g,
                           const StageScale &sc, cudaStream_t st)
{
    dim3 blocks((g.Wo + kTileW - 1) / kTileW, (g.Ho + kTileH - 1) / kTileH, g.N);
    const bool border = g.padding == PWS_PAD_BORDER, align = g.align != 0;
#define PWS_B(CS, GIN) do { \
        if (border && align) stages_bwd_kernel<T, G, CS, true, true, GIN><<<blocks, kThreads, 0, st>>>(in, sv, K, gin, g, sc); \
        else if (border) stages_bwd_kernel<T, G, CS, true, false, GIN><<<blocks, kThreads, 0, st>>>(in, sv, K, gin, g, sc); \
        else if (align) stages_bwd_kernel<T, G, CS, false, true, GIN><<<blocks, kThreads, 0, st>>>(in, sv, K, gin, g, sc); \
        else stages_bwd_kernel<T, G, CS, false, false, GIN><<<blocks, kThreads, 0, st>>>(in, sv, K, gin, g, sc); } while (0)
    if (g.C == 3) { if (want_gin) PWS_B(3, true); else PWS_B(3, false); }
    else { if (want_gin) PWS_B(1, true); else PWS_B(1, false); }
#undef PWS_B
}

// (frame, map) dtype -> instantiation; the host has already checked the pair (capi.cu)
template <typename F>
bool dispatch_types(int in_dtype, int map_dtype, F &&f)
{
    const bool same = map_dtype == in_dtype;
    if (in_dtype == PWS_F32 && same) f(float(), float());
    else if (in_dtype == PWS_F16 && same) f(__half(), __half());
    else if (in_dtype == PWS_F16 && map_dtype == PWS_F32) f(__half(), float());
    else if (in_dtype == PWS_BF16 && same) f(__nv_bfloat16(), __nv_bfloat16());
    else if (in_dtype == PWS_BF16 && map_dtype == PWS_F32) f(__nv_bfloat16(), float());
    else return false;
    return true;
}

}  // namespace

int launch_stages_forward(const View &in, int in_dtype, const StageViews &sv, int map_dtype, int K, const Geometry &g,
                          const StageScale &sc, cudaStream_t st)
{
    if (g.N > 65535 || (g.Ho + kTileH - 1) / kTileH > 65535) { set_error("stages forward: batch or height too large"); return PWS_EUNSUPPORTED; }
    if (g.C != 3 && g.C != 1) { set_error("stages forward: C must be 1 or 3 (got %d)", g.C); return PWS_EUNSUPPORTED; }
    const bool ok = dispatch_types(in_dtype, map_dtype, [&](auto t, auto m) {
        stages_forward_typed<decltype(t), decltype(m)>(in, sv, K, g, sc, st);
    });
    if (!ok) { set_error("stages forward: unsupported frame / map dtype pair (%d, %d)", in_dtype, map_dtype); return PWS_EUNSUPPORTED; }
    note_launch();
    note_kernel(in_dtype == PWS_F32 ? "stages_fwd" : "stages_fwd_16");
    return PWS_OK;
}

int launch_stages_backward(const View &in, int in_dtype, const StageViews &sv, int map_dtype, int K, const View &gin, bool want_gin,
                           const Geometry &g, const StageScale &sc, cudaStream_t st)
{
    if (g.N > 65535 || (g.Ho + kTileH - 1) / kTileH > 65535) { set_error("stages backward: batch or height too large"); return PWS_EUNSUPPORTED; }
    if (g.C != 3 && g.C != 1) { set_error("stages backward: C must be 1 or 3 (got %d)", g.C); return PWS_EUNSUPPORTED; }
    if (want_gin) {   // fp32 for every frame type: 16-bit frames accumulate into an f32 buffer
        cudaError_t e = cudaMemsetAsync(gin.p, 0, (size_t)g.N * g.C * g.H * g.W * sizeof(float), st);
        if (e != cudaSuccess) { set_error("stages backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
    }
    const bool ok = dispatch_types(in_dtype, map_dtype, [&](auto t, auto m) {
        stages_backward_typed<decltype(t), decltype(m)>(in, sv, K, gin, want_gin, g, sc, st);
    });
    if (!ok) { set_error("stages backward: unsupported frame / map dtype pair (%d, %d)", in_dtype, map_dtype); return PWS_EUNSUPPORTED; }
    note_launch();
    note_kernel(in_dtype == PWS_F32 ? "stages_bwd" : "stages_bwd_16");
    return PWS_OK;
}

}  // namespace pws
