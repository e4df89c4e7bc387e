// pws_common.cuh -- shared device helpers of libpwswarp (sm_100a).
//
// Coordinate pipeline of the pixel-wise warp, written with explicit rounding
// intrinsics so nvcc's contraction choices cannot drift from ATen's CUDA kernel
// ($TORCH/include/ATen/native/cuda/GridSampler.cuh:21-57,138-227; SASS order
// documented in SURVEY.md section 7): the fp32 path is bit-identical to torch.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <limits.h>

#include "../../include/pwswarp.h"

namespace pws {

// A strided 4-D view as the kernels see it. Within-frame offsets are 32-bit
// (validated on the host: one frame spans < 2^31 elements); the batch stride is 64-bit.
struct View {
    void *p;
    int64_t sN;
    int32_t s1, s2, s3;  // (C,H,W) strides for frames; (Ho,Wo,coord) strides for maps
};

struct Geometry {
    int32_t N, C, H, W;  // frame
    int32_t Ho, Wo;      // output / map
    int32_t padding;     // PWS_PAD_ZEROS | PWS_PAD_BORDER
    int32_t align;
};

// ---- element conversion -----------------------------------------------------------
template <typename T> struct Acc { using type = float; };
template <> struct Acc<double> { using type = double; };

template <typename T> __device__ __forceinline__ typename Acc<T>::type to_acc(T v) { return (typename Acc<T>::type)v; }
template <> __device__ __forceinline__ float to_acc<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_acc<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T, typename A> __device__ __forceinline__ T from_acc(A v) { return (T)v; }
template <> __device__ __forceinline__ __half from_acc<__half, float>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_acc<__nv_bfloat16, float>(float v) { return __float2bfloat16_rn(v); }

template <typename T> __device__ __forceinline__ T ldg(const T *p) { return __ldg(p); }

// one map pixel's (x, y) as a single vector access: 8 bytes for fp32 maps, 4 for 16-bit maps
__device__ __forceinline__ float2 ldg_pair(const float *p) { return __ldg(reinterpret_cast<const float2 *>(p)); }
__device__ __forceinline__ float2 ldg_pair(const __half *p) { return __half22float2(__ldg(reinterpret_cast<const __half2 *>(p))); }
__device__ __forceinline__ float2 ldg_pair(const __nv_bfloat16 *p) { return __bfloat1622float2(__ldg(reinterpret_cast<const __nv_bfloat162 *>(p))); }
__device__ __forceinline__ void st_pair(float *p, float x, float y) { *reinterpret_cast<float2 *>(p) = make_float2(x, y); }
__device__ __forceinline__ void st_pair(__half *p, float x, float y) { *reinterpret_cast<__half2 *>(p) = __floats2half2_rn(x, y); }
__device__ __forceinline__ void st_pair(__nv_bfloat16 *p, float x, float y) { *reinterpret_cast<__nv_bfloat162 *>(p) = __floats2bfloat162_rn(x, y); }

// ---- fp32 coordinate math, explicit rounding ----------------------------------------
__device__ __forceinline__ float unnormalize(float coord, int size, bool align)
{
    float t = __fadd_rn(coord, 1.0f);
    if (align) return __fmul_rn(__fmul_rn(t, 0.5f), (float)(size - 1));
    return __fmul_rn(__fmaf_rn(t, (float)size, -1.0f), 0.5f);
}
__device__ __forceinline__ double unnormalize(double coord, int size, bool align)
{
    if (align) return ((coord + 1.0) / 2.0) * (size - 1);
    return ((coord + 1.0) * size - 1.0) / 2.0;
}

__device__ __forceinline__ float safe_downgrade(float x)
{
    // INT_MAX-1 promotes to 2147483648.0f, exactly as in ATen's comparison
    if (x > (float)(INT_MAX - 1) || x < (float)INT_MIN || !isfinite(x)) return -100.0f;
    return x;
}
__device__ __forceinline__ double safe_downgrade(double x)
{
    if (x > (double)(INT_MAX - 1) || x < (double)INT_MIN || !isfinite(x)) return -100.0;
    return x;
}

// forward source index: unnormalise, clip for border padding (min/max drop a NaN), guard
template <typename A>
__device__ __forceinline__ A source_index(A coord, int size, int padding, bool align)
{
    A c = unnormalize(coord, size, align);
    if (padding == PWS_PAD_BORDER) c = min((A)(size - 1), max(c, (A)0));
    return safe_downgrade(c);
}

// backward source index: also d(index)/d(coord); borders are out of bounds for the gradient
template <typename A>
__device__ __forceinline__ A source_index_set_grad(A coord, int size, int padding, bool align, A *g)
{
    A c = unnormalize(coord, size, align);
    A gm = align ? (A)(size - 1) / 2 : (A)size / 2;
    if (padding == PWS_PAD_BORDER) {
        if (c <= (A)0) { c = (A)0; gm = gm * (A)0; }
        else {
            A mx = (A)(size - 1);
            if (c >= mx) { c = mx; gm = gm * (A)0; }
        }
    }
    *g = gm;
    return safe_downgrade(c);
}

// the four bilinear taps of one output pixel
template <typename A>
struct Taps {
    int x0, y0;
    A nw, ne, sw, se;
    A ix, iy;
    unsigned mask;  // bit0 nw, bit1 ne, bit2 sw, bit3 se
};

__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double fsub(double a, double b) { return a - b; }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double fmul(double a, double b) { return a * b; }
__device__ __forceinline__ float ffma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ double ffma(double a, double b, double c) { return fma(a, b, c); }

template <typename A>
__device__ __forceinline__ void make_taps(A ix, A iy, int H, int W, Taps<A> &t)
{
    int x0 = (int)floor(ix), y0 = (int)floor(iy);
    A x0f = (A)x0, y0f = (A)y0, x1f = (A)(x0 + 1), y1f = (A)(y0 + 1);
    A wx0 = fsub(x1f, ix), wx1 = fsub(ix, x0f), wy0 = fsub(y1f, iy), wy1 = fsub(iy, y0f);
    t.x0 = x0; t.y0 = y0; t.ix = ix; t.iy = iy;
    t.nw = fmul(wx0, wy0);
    t.ne = fmul(wx1, wy0);
    t.sw = fmul(wx0, wy1);
    t.se = fmul(wx1, wy1);
    // unsigned compares fold the two-sided range checks
    bool xw = (unsigned)x0 < (unsigned)W, xe = (unsigned)(x0 + 1) < (unsigned)W;
    bool yn = (unsigned)y0 < (unsigned)H, ys = (unsigned)(y0 + 1) < (unsigned)H;
    t.mask = ((xw && yn) ? 1u : 0u) | ((xe && yn) ? 2u : 0u) | ((xw && ys) ? 4u : 0u) | ((xe && ys) ? 8u : 0u);
}

// The lean kernels access an interleaved map (s3 == 1) one (x, y) pair per pixel (ldg_pair / st_pair), which needs every
// pixel's pair aligned to its size; planar maps take scalar accesses and always qualify.
inline bool map_pairs_ok(const View &v, int elem_bytes)
{
    return v.s3 != 1 || (!(reinterpret_cast<uintptr_t>(v.p) & (uintptr_t)(2 * elem_bytes - 1)) && !(v.sN & 1) && !(v.s1 & 1) &&
                         !(v.s2 & 1));
}

// ---- error plumbing (host) -----------------------------------------------------------
void set_error(const char *fmt, ...);
void note_launch(int kernels = 1);  // bumps the counter pws_launch_count() reports
void note_kernel(const char *family);  // what pws_last_kernel() reports (thread-local)

struct Problem {  // validated, kernel-ready description of one call
    Geometry g;
    View in, grid, out;       // forward
    View gout, gin, ggrid;    // backward
    int in_dtype, grid_dtype;
    bool want_gin, want_ggrid;
};

struct MapSpec {  // kernel-side form of pws_map_spec (warp_fused.cu)
    View drift;          // (N, mh, mw, 2) of drift_dtype; p == nullptr: zero drift
    const float *theta;  // (N,2,3) for the affine base
    int base;            // PWS_BASE_*
    int base_align;      // align_corners of affine_grid
    int upsample;        // PWS_UP_*
    int mh, mw;          // map lattice size
    float pre_add, pre_mul, post_div, post_add;
    int has_pre, has_post;
    int drift_dtype;     // PWS_F32 / PWS_F16 / PWS_BF16 (host dispatch only)
};

// K maps applied to one frame (warp_stages.cu)
constexpr int kMaxStages = 4;
struct StageViews {
    View map[kMaxStages];
    View io[kMaxStages];     // forward: outputs; backward: grad_outputs
    View gg[kMaxStages];     // backward: grad_grids (p == nullptr: not wanted)
};
struct StageScale {
    float pre_add, pre_mul, post_mul, post_add;
    int has_pre, has_post;
};
// in_dtype: f32 / f16 / bf16; map_dtype: f32 or in_dtype (one dtype for all K maps); gin is f32 for every frame type
int launch_stages_forward(const View &in, int in_dtype, const StageViews &sv, int map_dtype, int K, const Geometry &g,
                          const StageScale &sc, cudaStream_t st);
int launch_stages_backward(const View &in, int in_dtype, const StageViews &sv, int map_dtype, int K, const View &gin, bool want_gin,
                           const Geometry &g, const StageScale &sc, cudaStream_t st);

// Calls whose whole working set sits in L2 (the reference's training shapes: 16 x 3 x 256 x 256 = 12.6 MB) are bound by the
// launch, not by HBM: they take the plain one-wave kernels (no tensor maps to encode, no counter slot to lease, no
// 227 KB persistent CTAs to set up) instead of the TMA pipelines.
#ifndef PWS_SMALL_ELEMS
#define PWS_SMALL_ELEMS (4 << 20)   // output elements (16 MB of fp32): default of pws_small_problem_elems()
#endif
int64_t small_problem_threshold();   // capi.cu
inline bool small_problem(const Problem &pb)
{
    return (int64_t)pb.g.N * pb.g.C * pb.g.Ho * pb.g.Wo <= small_problem_threshold();
}

int launch_forward(const Problem &pb, cudaStream_t st);
int launch_backward(const Problem &pb, cudaStream_t st);
int launch_taps(const View &grid, const Geometry &g, int32_t *x0, int32_t *y0, uint8_t *mask, float *w, cudaStream_t st);

}  // namespace pws
