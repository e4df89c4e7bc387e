/*
 * oracle/warp_oracle.c -- CPU restatement of the pixel-wise bilinear warp.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under pwstablenet_b200/ may import, link
 * or execute this file; it is the checker for tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline leg, never the product path.
 *
 * The reference (mindazhao/PWStableNet) holds no arithmetic of its own for
 * this path: it calls torch.nn.functional.grid_sample at
 *   R/main_new.py:106,109,116,118,197,716   (R = /root/reference)
 * and builds the maps at
 *   R/lib/networks_cascading.py:164,174,235   (tanh drift + affine_grid)
 *   R/lib/utils.py:386-403                    (generate_maps: drift + identity)
 *   R/main_new.py:706-710                     (UpsamplingBilinear2d of the map)
 * The algorithm therefore lives in a third-party dependency, PyTorch/ATen
 * (reference pin "pytorch 0.4.0+", R/README.md:27; this image: 2.11.0+cu128).
 * What follows restates ATen's published algorithm from the shipped headers
 *   $TORCH/include/ATen/native/cuda/GridSampler.cuh:21-57,138-227,248-262
 *   $TORCH/include/ATen/native/GridSampler.h:26-276
 *   $TORCH/include/ATen/native/cuda/UpSample.cuh:96-130
 * with the floating-point operation ORDER of the CUDA kernel (single-rounded
 * fma in the unnormalise step, products by multiply, tap accumulation by fma
 * in the order nw, ne, sw, se), so that a GPU kernel following the same order
 * is bit-identical to this file.
 *
 * Parity pin: tests/golden/ holds vectors produced by running the reference's
 * own netG (imported from /root/reference) and torch's CPU grid_sample in the
 * build container (tests/golden/make_golden.py); tests/test_oracle_golden.py
 * checks this file against them.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared (see oracle/Makefile).  Contraction is
 * disabled so that only the explicit fmaf() calls fuse.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <limits.h>

#define ORACLE_API __attribute__((visibility("default")))

/* ---- coordinate pipeline (GridSampler.cuh:21-57,138-180) -------------------- */

/* grid_sampler_unnormalize: [-1,1] -> pixel index.  nvcc emits
 *   align_corners : FADD(x,1) ; FMUL 0.5 ; FMUL (size-1)
 *   otherwise     : FADD(x,1) ; FFMA(.,size,-1) ; FMUL 0.5
 * (SURVEY.md section 7 "hard parts": SASS offsets 0x700-0x740). */
static inline float unnormalize_f32(float coord, int size, int align)
{
    float t = coord + 1.0f;
    if (align)
        return (t * 0.5f) * (float)(size - 1);
    return fmaf(t, (float)size, -1.0f) * 0.5f;
}

/* clip_coordinates (forward, GridSampler.cuh:53-57): min(size-1, max(in, 0)),
 * with CUDA fmaxf/fminf NaN behaviour (NaN operand is dropped). */
static inline float clip_f32(float in, int size)
{
    return fminf((float)(size - 1), fmaxf(in, 0.0f));
}

/* clip_coordinates_set_grad (backward, GridSampler.cuh:62-80): borders count
 * as out of bounds for the gradient. */
static inline float clip_set_grad_f32(float in, int size, float *g)
{
    if (in <= 0.0f) { *g = 0.0f; return 0.0f; }
    float mx = (float)(size - 1);
    if (in >= mx) { *g = 0.0f; return mx; }
    *g = 1.0f;
    return in;
}

/* safe_downgrade_to_int_range (GridSampler.cuh:138-147). INT_MAX-1 promotes
 * to float 2147483648.0f in the comparison, as it does under nvcc. */
static inline float safe_downgrade_f32(float x)
{
    if (x > (float)(INT_MAX - 1) || x < (float)INT_MIN || !isfinite((double)x))
        return -100.0f;
    return x;
}

/* padding: 0 zeros, 1 border (reflection = 2 is out of scope: SURVEY 8(b)) */
static inline float source_index_f32(float coord, int size, int padding, int align)
{
    float c = unnormalize_f32(coord, size, align);
    if (padding == 1) c = clip_f32(c, size);
    return safe_downgrade_f32(c);
}

static inline float source_index_set_grad_f32(float coord, int size, int padding,
                                              int align, float *g)
{
    float c = unnormalize_f32(coord, size, align);
    *g = align ? (float)(size - 1) / 2.0f : (float)size / 2.0f;
    if (padding == 1) {
        float gc;
        c = clip_set_grad_f32(c, size, &gc);
        *g = (*g) * gc;
    }
    return safe_downgrade_f32(c);
}

static inline int in_bounds(int y, int x, int H, int W)
{
    return y >= 0 && y < H && x >= 0 && x < W;
}

typedef struct {
    int x0, y0;            /* north-west tap */
    float nw, ne, sw, se;  /* weights */
    float ix, iy;          /* source index after padding */
    unsigned mask;         /* bit0 nw, bit1 ne, bit2 sw, bit3 se in bounds */
} taps_t;

static inline void make_taps(float ix, float iy, int H, int W, taps_t *t)
{
    int x0 = (int)floorf(ix), y0 = (int)floorf(iy);
    float x1f = (float)(x0 + 1), y1f = (float)(y0 + 1);
    float x0f = (float)x0, y0f = (float)y0;
    t->x0 = x0; t->y0 = y0; t->ix = ix; t->iy = iy;
    t->nw = (x1f - ix) * (y1f - iy);
    t->ne = (ix - x0f) * (y1f - iy);
    t->sw = (x1f - ix) * (iy - y0f);
    t->se = (ix - x0f) * (iy - y0f);
    t->mask = (in_bounds(y0, x0, H, W) ? 1u : 0u) | (in_bounds(y0, x0 + 1, H, W) ? 2u : 0u) |
              (in_bounds(y0 + 1, x0, H, W) ? 4u : 0u) | (in_bounds(y0 + 1, x0 + 1, H, W) ? 8u : 0u);
}

/* ---- taps debug (what pws_warp2d_taps returns) ------------------------------ */

ORACLE_API void oracle_warp2d_taps_f32(
    const float *grid, const int64_t gstride[4], /* (N,Ho,Wo,2) element strides */
    int N, int Ho, int Wo, int H, int W, int padding, int align,
    int32_t *x0, int32_t *y0, uint8_t *mask, float *weights /* nullable, (N,Ho,Wo,4) */)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < Ho; ++h)
            for (int w = 0; w < Wo; ++w) {
                const float *g = grid + n * gstride[0] + h * gstride[1] + w * gstride[2];
                float ix = source_index_f32(g[0], W, padding, align);
                float iy = source_index_f32(g[gstride[3]], H, padding, align);
                taps_t t; make_taps(ix, iy, H, W, &t);
                int64_t o = ((int64_t)n * Ho + h) * Wo + w;
                x0[o] = t.x0; y0[o] = t.y0; mask[o] = (uint8_t)t.mask;
                if (weights) {
                    weights[4 * o + 0] = t.nw; weights[4 * o + 1] = t.ne;
                    weights[4 * o + 2] = t.sw; weights[4 * o + 3] = t.se;
                }
            }
}

/* ---- forward (R/main_new.py:106,116,197,716 -> grid_sampler_2d) --------------- */

ORACLE_API void oracle_warp2d_forward_f32(
    const float *in, const int64_t istride[4],   /* (N,C,H,W) */
    const float *grid, const int64_t gstride[4], /* (N,Ho,Wo,2) */
    float *out, const int64_t ostride[4],        /* (N,C,Ho,Wo) */
    int N, int C, int H, int W, int Ho, int Wo, int padding, int align)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < Ho; ++h)
            for (int w = 0; w < Wo; ++w) {
                const float *g = grid + n * gstride[0] + h * gstride[1] + w * gstride[2];
                float ix = source_index_f32(g[0], W, padding, align);
                float iy = source_index_f32(g[gstride[3]], H, padding, align);
                taps_t t; make_taps(ix, iy, H, W, &t);
                for (int c = 0; c < C; ++c) {
                    const float *p = in + n * istride[0] + c * istride[1];
                    float acc = 0.0f;
                    if (t.mask & 1u) acc = fmaf(p[t.y0 * istride[2] + t.x0 * istride[3]], t.nw, acc);
                    if (t.mask & 2u) acc = fmaf(p[t.y0 * istride[2] + (t.x0 + 1) * istride[3]], t.ne, acc);
                    if (t.mask & 4u) acc = fmaf(p[(t.y0 + 1) * istride[2] + t.x0 * istride[3]], t.sw, acc);
                    if (t.mask & 8u) acc = fmaf(p[(t.y0 + 1) * istride[2] + (t.x0 + 1) * istride[3]], t.se, acc);
                    out[n * ostride[0] + c * ostride[1] + h * ostride[2] + w * ostride[3]] = acc;
                }
            }
}

/* ---- backward (autograd of the above, R/main_new.py:214) ---------------------
 * grad_in is accumulated sequentially in (n,h,w,c,tap) order: deterministic,
 * one of the orders the GPU's atomics may realise.  grad_in_f64, when given,
 * receives the same sums accumulated in double (the order-free truth the
 * 1e-4 relative tolerance is measured against).  Both must arrive zeroed. */
ORACLE_API void oracle_warp2d_backward_f32(
    const float *gout, const int64_t gostride[4], /* (N,C,Ho,Wo) */
    const float *in, const int64_t istride[4],
    const float *grid, const int64_t gstride[4],
    float *grad_in,      /* nullable; contiguous (N,C,H,W) */
    double *grad_in_f64, /* nullable; contiguous (N,C,H,W) */
    float *grad_grid,    /* nullable; contiguous (N,Ho,Wo,2) */
    int N, int C, int H, int W, int Ho, int Wo, int padding, int align)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < Ho; ++h)
            for (int w = 0; w < Wo; ++w) {
                const float *g = grid + n * gstride[0] + h * gstride[1] + w * gstride[2];
                float gxm, gym;
                float ix = source_index_set_grad_f32(g[0], W, padding, align, &gxm);
                float iy = source_index_set_grad_f32(g[gstride[3]], H, padding, align, &gym);
                taps_t t; make_taps(ix, iy, H, W, &t);
                float x0f = (float)t.x0, y0f = (float)t.y0;
                float x1f = (float)(t.x0 + 1), y1f = (float)(t.y0 + 1);
                float gix = 0.0f, giy = 0.0f;
                for (int c = 0; c < C; ++c) {
                    float go = gout[n * gostride[0] + c * gostride[1] + h * gostride[2] + w * gostride[3]];
                    const float *p = in + n * istride[0] + c * istride[1];
                    int64_t plane = ((int64_t)n * C + c) * H * W;
                    const int ty[4] = { t.y0, t.y0, t.y0 + 1, t.y0 + 1 };
                    const int tx[4] = { t.x0, t.x0 + 1, t.x0, t.x0 + 1 };
                    const float tw[4] = { t.nw, t.ne, t.sw, t.se };
                    for (int k = 0; k < 4; ++k)
                        if (t.mask & (1u << k)) {
                            int64_t o = plane + (int64_t)ty[k] * W + tx[k];
                            if (grad_in) grad_in[o] += tw[k] * go;
                            if (grad_in_f64) grad_in_f64[o] += (double)tw[k] * (double)go;
                        }
                    if (grad_grid) {
                        /* order and contraction as nvcc compiles the upstream body:
                         *   gix -= v * (y1 - iy) * gOut  ->  t = v*(y1-iy); gix = fma(-t, gOut, gix) */
                        if (t.mask & 1u) {
                            float v = p[t.y0 * istride[2] + t.x0 * istride[3]];
                            gix = fmaf(-(v * (y1f - iy)), go, gix);
                            giy = fmaf(-(v * (x1f - ix)), go, giy);
                        }
                        if (t.mask & 2u) {
                            float v = p[t.y0 * istride[2] + (t.x0 + 1) * istride[3]];
                            gix = fmaf(v * (y1f - iy), go, gix);
                            giy = fmaf(-(v * (ix - x0f)), go, giy);
                        }
                        if (t.mask & 4u) {
                            float v = p[(t.y0 + 1) * istride[2] + t.x0 * istride[3]];
                            gix = fmaf(-(v * (iy - y0f)), go, gix);
                            giy = fmaf(v * (x1f - ix), go, giy);
                        }
                        if (t.mask & 8u) {
                            float v = p[(t.y0 + 1) * istride[2] + (t.x0 + 1) * istride[3]];
                            gix = fmaf(v * (iy - y0f), go, gix);
                            giy = fmaf(v * (ix - x0f), go, giy);
                        }
                    }
                }
                if (grad_grid) {
                    int64_t o = (((int64_t)n * Ho + h) * Wo + w) * 2;
                    grad_grid[o] = gxm * gix;
                    grad_grid[o + 1] = gym * giy;
                }
            }
}

/* ---- double-precision twins (gradcheck-grade truth; plain arithmetic) -------- */

static inline double source_index_f64(double coord, int size, int padding, int align, double *g)
{
    double c, gm;
    if (align) { c = ((coord + 1.0) / 2.0) * (size - 1); gm = (double)(size - 1) / 2.0; }
    else       { c = ((coord + 1.0) * size - 1.0) / 2.0; gm = (double)size / 2.0; }
    if (padding == 1) {
        if (g) {
            if (c <= 0.0) { c = 0.0; gm = 0.0; }
            else if (c >= (double)(size - 1)) { c = (double)(size - 1); gm = 0.0; }
        } else {
            c = fmin((double)(size - 1), fmax(c, 0.0));
        }
    }
    if (c > (double)(INT_MAX - 1) || c < (double)INT_MIN || !isfinite(c)) c = -100.0;
    if (g) *g = gm;
    return c;
}

ORACLE_API void oracle_warp2d_forward_f64(
    const double *in, const int64_t istride[4], const double *grid, const int64_t gstride[4],
    double *out, const int64_t ostride[4],
    int N, int C, int H, int W, int Ho, int Wo, int padding, int align)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < Ho; ++h)
            for (int w = 0; w < Wo; ++w) {
                const double *g = grid + n * gstride[0] + h * gstride[1] + w * gstride[2];
                double ix = source_index_f64(g[0], W, padding, align, 0);
                double iy = source_index_f64(g[gstride[3]], H, padding, align, 0);
                int x0 = (int)floor(ix), y0 = (int)floor(iy);
                double wx1 = ix - x0, wx0 = (x0 + 1) - ix, wy1 = iy - y0, wy0 = (y0 + 1) - iy;
                for (int c = 0; c < C; ++c) {
                    const double *p = in + n * istride[0] + c * istride[1];
                    double acc = 0.0;
                    if (in_bounds(y0, x0, H, W)) acc += p[y0 * istride[2] + x0 * istride[3]] * (wx0 * wy0);
                    if (in_bounds(y0, x0 + 1, H, W)) acc += p[y0 * istride[2] + (x0 + 1) * istride[3]] * (wx1 * wy0);
                    if (in_bounds(y0 + 1, x0, H, W)) acc += p[(y0 + 1) * istride[2] + x0 * istride[3]] * (wx0 * wy1);
                    if (in_bounds(y0 + 1, x0 + 1, H, W)) acc += p[(y0 + 1) * istride[2] + (x0 + 1) * istride[3]] * (wx1 * wy1);
                    out[n * ostride[0] + c * ostride[1] + h * ostride[2] + w * ostride[3]] = acc;
                }
            }
}

ORACLE_API void oracle_warp2d_backward_f64(
    const double *gout, const int64_t gostride[4], const double *in, const int64_t istride[4],
    const double *grid, const int64_t gstride[4],
    double *grad_in /* nullable, zeroed, contiguous */, double *grad_grid /* nullable, contiguous */,
    int N, int C, int H, int W, int Ho, int Wo, int padding, int align)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < Ho; ++h)
            for (int w = 0; w < Wo; ++w) {
                const double *g = grid + n * gstride[0] + h * gstride[1] + w * gstride[2];
                double gxm, gym;
                double ix = source_index_f64(g[0], W, padding, align, &gxm);
                double iy = source_index_f64(g[gstride[3]], H, padding, align, &gym);
                int x0 = (int)floor(ix), y0 = (int)floor(iy);
                double wx1 = ix - x0, wx0 = (x0 + 1) - ix, wy1 = iy - y0, wy0 = (y0 + 1) - iy;
                double gix = 0.0, giy = 0.0;
                for (int c = 0; c < C; ++c) {
                    double go = gout[n * gostride[0] + c * gostride[1] + h * gostride[2] + w * gostride[3]];
                    const double *p = in + n * istride[0] + c * istride[1];
                    int64_t plane = ((int64_t)n * C + c) * H * W;
                    if (in_bounds(y0, x0, H, W)) {
                        double v = p[y0 * istride[2] + x0 * istride[3]];
                        if (grad_in) grad_in[plane + (int64_t)y0 * W + x0] += wx0 * wy0 * go;
                        gix -= v * wy0 * go; giy -= v * wx0 * go;
                    }
                    if (in_bounds(y0, x0 + 1, H, W)) {
                        double v = p[y0 * istride[2] + (x0 + 1) * istride[3]];
                        if (grad_in) grad_in[plane + (int64_t)y0 * W + x0 + 1] += wx1 * wy0 * go;
                        gix += v * wy0 * go; giy -= v * wx1 * go;
                    }
                    if (in_bounds(y0 + 1, x0, H, W)) {
                        double v = p[(y0 + 1) * istride[2] + x0 * istride[3]];
                        if (grad_in) grad_in[plane + (int64_t)(y0 + 1) * W + x0] += wx0 * wy1 * go;
                        gix -= v * wy1 * go; giy += v * wx0 * go;
                    }
                    if (in_bounds(y0 + 1, x0 + 1, H, W)) {
                        double v = p[(y0 + 1) * istride[2] + (x0 + 1) * istride[3]];
                        if (grad_in) grad_in[plane + (int64_t)(y0 + 1) * W + x0 + 1] += wx1 * wy1 * go;
                        gix += v * wy1 * go; giy += v * wx1 * go;
                    }
                }
                if (grad_grid) {
                    int64_t o = (((int64_t)n * Ho + h) * Wo + w) * 2;
                    grad_grid[o] = gxm * gix;
                    grad_grid[o + 1] = gym * giy;
                }
            }
}

/* ---- map composition ---------------------------------------------------------- */

/* generate_maps (R/lib/utils.py:386-403): map = drift + identity meshgrid in the
 * align_corners=True convention, X*2/(W-1)-1 evaluated as torch does on float
 * tensors: (X*2) [exact], IEEE divide by (W-1), subtract 1.  Planar (N,2,H,W)
 * in and out; channel 0 = x, channel 1 = y. */
ORACLE_API void oracle_generate_maps_f32(const float *drift, float *map, int N, int H, int W)
{
    for (int n = 0; n < N; ++n)
        for (int h = 0; h < H; ++h)
            for (int w = 0; w < W; ++w) {
                float bx = ((float)w * 2.0f) / (float)(W - 1) - 1.0f;
                float by = ((float)h * 2.0f) / (float)(H - 1) - 1.0f;
                int64_t o = (((int64_t)n * 2) * H + h) * W + w;
                map[o] = drift[o] + bx;
                map[o + (int64_t)H * W] = drift[o + (int64_t)H * W] + by;
            }
}

/* affine_grid base coordinate (aten::affine_grid_generator -> linspace):
 * linspace(-1,1,S)[i] is evaluated by ATen as start + step*i for i < S/2 and
 * end - step*(S-1-i) otherwise, step = 2/(S-1); when !align_corners the result
 * is multiplied by (S-1)/S. */
static inline float affine_base_f32(int i, int S, int align)
{
    if (S <= 1) return 0.0f;
    float step = 2.0f / (float)(S - 1);
    float v = (i < S / 2) ? fmaf(step, (float)i, -1.0f) : fmaf(-step, (float)(S - 1 - i), 1.0f); /* contracted, as on the GPU */
    if (!align) v = v * (float)(S - 1) / (float)S;
    return v;
}

/* map = drift (planar N,2,H,W; may be NULL) + affine_grid(theta (N,2,3)).
 * R/lib/networks_cascading.py:164,235.  The product with theta is a K=3 dot
 * product, here x*t0 + y*t1 + t2 in that order by fma; torch's bmm may order
 * it differently, so this function is held to a 1-ulp-of-the-map tolerance
 * (DESIGN.md "fused composition contract"), not to bit equality. Output is
 * interleaved (N,H,W,2). */
ORACLE_API void oracle_affine_map_f32(const float *theta, const float *drift, float *map,
                                      int N, int H, int W, int align)
{
    for (int n = 0; n < N; ++n) {
        const float *t = theta + n * 6;
        for (int h = 0; h < H; ++h)
            for (int w = 0; w < W; ++w) {
                float bx = affine_base_f32(w, W, align), by = affine_base_f32(h, H, align);
                float mx = fmaf(bx, t[0], fmaf(by, t[1], t[2]));
                float my = fmaf(bx, t[3], fmaf(by, t[4], t[5]));
                if (drift) {
                    int64_t o = (((int64_t)n * 2) * H + h) * W + w;
                    mx = drift[o] + mx;
                    my = drift[o + (int64_t)H * W] + my;
                }
                int64_t o2 = (((int64_t)n * H + h) * W + w) * 2;
                map[o2] = mx; map[o2 + 1] = my;
            }
    }
}

/* ---- the map upsample (UpSample.cuh:96-130) and its adjoint ------------------- */

/* Source scale of upsample_bilinear2d: (src-1)/(dst-1) aligned (0 for a 1-pixel
 * destination), src/dst otherwise; one IEEE division, as on the GPU. */
static inline float up_scale_f32(int src, int dst, int align)
{
    if (align) return dst > 1 ? (float)(src - 1) / (float)(dst - 1) : 0.0f;
    return (float)src / (float)dst;
}

typedef struct { int i0, ip; float l0, l1; } up_coef_t;

/* Source index of destination index dst: one fp32 multiply aligned, one fma
 * half_pixel (clamped at 0); lambdas l1 = s - i0, l0 = 1 - l1. */
static inline up_coef_t up_coef_f32(int dst, int src, float scale, int align)
{
    float s = align ? scale * (float)dst : fmaf(scale, (float)dst + 0.5f, -0.5f);
    if (!align && s < 0.0f) s = 0.0f;
    up_coef_t c;
    c.i0 = (int)s;
    c.ip = (c.i0 < src - 1) ? 1 : 0;
    c.l1 = s - (float)c.i0;
    c.l0 = 1.0f - c.l1;
    return c;
}

/* The coefficients of destination indices 0..dst-1 from a source of size src
 * (what the backward's tile census restates). */
ORACLE_API void oracle_upsample_coefs_f32(int src, int dst, int align, int32_t *i0, int32_t *ip,
                                          float *l0, float *l1)
{
    const float r = up_scale_f32(src, dst, align);
    for (int d = 0; d < dst; ++d) {
        up_coef_t c = up_coef_f32(d, src, r, align);
        i0[d] = c.i0; ip[d] = c.ip; l0[d] = c.l0; l1[d] = c.l1;
    }
}

/* Bilinear resize of a planar map (N,2,h,w) -> (N,2,H,W), the map upsample of
 * R/main_new.py:706-710 (UpsamplingBilinear2d: align_corners=True) and
 * R/main.py:639-641 (nn.Upsample bilinear: align_corners=False).
 * Blend order as upsample_bilinear2d_out_frame:
 *   h0lambda*(w0lambda*v00 + w1lambda*v01) + h1lambda*(w0lambda*v10 + w1lambda*v11)
 * with nvcc contraction: inner = fma(w0l, v00, w1l*v01), outer = fma(h0l, top, h1l*bot). */
ORACLE_API void oracle_upsample_map_f32(const float *src, float *dst, int N, int h, int w,
                                        int H, int W, int align)
{
    const float rh = up_scale_f32(h, H, align), rw = up_scale_f32(w, W, align);
    for (int n = 0; n < N * 2; ++n)
        for (int y = 0; y < H; ++y) {
            const up_coef_t cy = up_coef_f32(y, h, rh, align);
            for (int x = 0; x < W; ++x) {
                const up_coef_t cx = up_coef_f32(x, w, rw, align);
                const float *p = src + (int64_t)n * h * w;
                float v00 = p[cy.i0 * w + cx.i0], v01 = p[cy.i0 * w + cx.i0 + cx.ip];
                float v10 = p[(cy.i0 + cy.ip) * w + cx.i0], v11 = p[(cy.i0 + cy.ip) * w + cx.i0 + cx.ip];
                float top = fmaf(cx.l0, v00, cx.l1 * v01);
                float bot = fmaf(cx.l0, v10, cx.l1 * v11);
                dst[((int64_t)n * H + y) * W + x] = fmaf(cy.l0, top, cy.l1 * bot);
            }
        }
}

/* Adjoint of oracle_upsample_map_f32 with its fp32 coefficients: the gradient gmap
 * (planar (N,2,H,W), fp64) of the upsampled map pushed to the lattice (N,2,h,w).
 * Every pixel hands each of the four nodes it blends the term t = h_l * w_l * g
 * (a node read twice, ip == 0, takes two terms).  Per node, in fp64: glat = sum t,
 * gabs = sum |t|, nterms = the number of terms.  All three must arrive zeroed. */
ORACLE_API void oracle_upsample_map_backward_f64(const double *gmap, int N, int h, int w, int H, int W, int align,
                                                 double *glat, double *gabs, int64_t *nterms)
{
    const float rh = up_scale_f32(h, H, align), rw = up_scale_f32(w, W, align);
    for (int n = 0; n < N * 2; ++n)
        for (int y = 0; y < H; ++y) {
            const up_coef_t cy = up_coef_f32(y, h, rh, align);
            for (int x = 0; x < W; ++x) {
                const up_coef_t cx = up_coef_f32(x, w, rw, align);
                const double g = gmap[((int64_t)n * H + y) * W + x];
                const int rows[2] = { cy.i0, cy.i0 + cy.ip }, cols[2] = { cx.i0, cx.i0 + cx.ip };
                const double hl[2] = { cy.l0, cy.l1 }, wl[2] = { cx.l0, cx.l1 };
                for (int a = 0; a < 2; ++a)
                    for (int b = 0; b < 2; ++b) {
                        const int64_t o = ((int64_t)n * h + rows[a]) * w + cols[b];
                        const double t = hl[a] * wl[b] * g;
                        glat[o] += t; gabs[o] += fabs(t); nterms[o] += 1;
                    }
            }
        }
}

/* d loss / d theta of the affine base: gtheta[n,c,:] = sum_ij glat[n,i,j,c] *
 * (bx_j, by_i, 1) with affine_base_f32's coordinates, in fp64; gabs the sums of
 * the terms' magnitudes.  glat interleaved (N,h,w,2); gtheta, gabs (N,2,3), zeroed. */
ORACLE_API void oracle_affine_theta_grad_f64(const double *glat, int N, int h, int w, int align,
                                             double *gtheta, double *gabs)
{
    for (int n = 0; n < N; ++n)
        for (int i = 0; i < h; ++i)
            for (int j = 0; j < w; ++j) {
                const double b[3] = { affine_base_f32(j, w, align), affine_base_f32(i, h, align), 1.0 };
                for (int c = 0; c < 2; ++c) {
                    const double g = glat[(((int64_t)n * h + i) * w + j) * 2 + c];
                    for (int k = 0; k < 3; ++k) {
                        gtheta[(n * 2 + c) * 3 + k] += g * b[k];
                        gabs[(n * 2 + c) * 3 + k] += fabs(g * b[k]);
                    }
                }
            }
}

ORACLE_API int oracle_abi_version(void) { return 2; }
