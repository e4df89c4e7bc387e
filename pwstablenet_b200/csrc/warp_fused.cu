// warp_fused.cu -- forward warp with the map composition fused into the sample.
//
// In the reference the map handed to grid_sample is itself the product of a few
// elementwise / resampling passes over HBM (SURVEY.md 0.4, 8(a) rows a7-a11):
//   a8  map = tanh-drift.permute(0,2,3,1) + affine_grid(theta)     R/lib/networks_cascading.py:164,235
//   a9  map = drift + identity meshgrid (generate_maps)             R/lib/utils.py:386-403
//   a10 map = bilinear upsample of the 256x256 map to the frame     R/main_new.py:706-710, R/main.py:639-641
//   a11 frame = (x+1)*127.5 before, out/127.5-1 after               R/main_new.py:106-107
//   a4  frame arrives as uint8 HWC from cv2 and leaves as uint8     R/main_new.py:679-684,717-721
// Here all of that happens in registers of the sampling kernel: the composed and
// upsampled map, the scaled frame and the fp32 output of the unfused pipeline are
// never written to HBM.  pws_compose_map emits the map the kernel uses, so tests can
// hold it to the torch-composed map and hold the fused sample to the plain sample of
// that very map (bit-exact).
//
// Generic strides (uint8 HWC frames and planar low-resolution drifts are the norm here),
// taps through L1, 4 pixels per thread as in the direct kernel.
// The backward (bwd_fused_kernel) recomputes the map with the same statements and takes the gradient to the frame, to the
// lattice through the upsample's adjoint, and (theta_grad_kernel) to theta of the affine base: the full-resolution map
// and its gradient never exist in HBM either.
#include "pws_common.cuh"

#include <type_traits>

namespace pws {

namespace {

__device__ __forceinline__ float lattice_base(int i, int S, int base, int align)
{
    if (base == PWS_BASE_IDENTITY)  // generate_maps: X*2/(S-1)-1 on float tensors
        return __fsub_rn(__fdiv_rn(__fmul_rn((float)i, 2.0f), (float)(S - 1)), 1.0f);
    // affine_grid's linspace(-1,1,S) (times (S-1)/S when not align_corners)
    if (S <= 1) return 0.0f;
    const float step = __fdiv_rn(2.0f, (float)(S - 1));
    float v = (i < S / 2) ? __fmaf_rn(step, (float)i, -1.0f) : __fmaf_rn(-step, (float)(S - 1 - i), 1.0f);  // as nvcc contracts ATen's linspace
    if (!align) v = __fdiv_rn(__fmul_rn(v, (float)(S - 1)), (float)S);
    return v;
}

// map value at lattice point (i, j) of item n:  drift + base.  L: the drift's element type (float, or the __half /
// __nv_bfloat16 lattice of a half-precision netG); the upcast is exact and everything after it is fp32.
template <typename L>
__device__ __forceinline__ void lattice_map(const MapSpec &m, int n, int i, int j, float &mx, float &my)
{
    float dx = 0.f, dy = 0.f;
    if (m.drift.p) {
        const L *d = (const L *)m.drift.p + (int64_t)n * m.drift.sN + i * m.drift.s1 + j * m.drift.s2;
        // interleaved (x,y) pairs -- the lattice the host side composes -- come as one 8-byte (fp32) or 4-byte (16-bit) load
        if (m.drift.s3 == 1 && !((reinterpret_cast<uintptr_t>(m.drift.p) & (2 * sizeof(L) - 1)) | ((m.drift.sN | m.drift.s1 | m.drift.s2) & 1))) {
            const float2 v = ldg_pair(d);
            dx = v.x; dy = v.y;
        } else {
            dx = to_acc(ldg(d)); dy = to_acc(ldg(d + m.drift.s3));
        }
    }
    if (m.base == PWS_BASE_NONE) { mx = dx; my = dy; return; }
    const float bx = lattice_base(j, m.mw, m.base, m.base_align), by = lattice_base(i, m.mh, m.base, m.base_align);
    if (m.base == PWS_BASE_IDENTITY) { mx = __fadd_rn(dx, bx); my = __fadd_rn(dy, by); return; }
    const float *t = m.theta + n * 6;
    const float ax = __fmaf_rn(bx, __ldg(t + 0), __fmaf_rn(by, __ldg(t + 1), __ldg(t + 2)));
    const float ay = __fmaf_rn(bx, __ldg(t + 3), __fmaf_rn(by, __ldg(t + 4), __ldg(t + 5)));
    mx = __fadd_rn(dx, ax); my = __fadd_rn(dy, ay);
}

struct UpCoef { int i0, ip; float l0, l1; };

// upsample_bilinear2d source index (UpSample.cuh:96-130)
__device__ __forceinline__ UpCoef up_coef(int dst, int src_size, float scale, bool align)
{
    float s = align ? __fmul_rn(scale, (float)dst) : __fmaf_rn(scale, __fadd_rn((float)dst, 0.5f), -0.5f);
    if (!align && s < 0.f) s = 0.f;
    UpCoef c;
    c.i0 = (int)s;
    c.ip = (c.i0 < src_size - 1) ? 1 : 0;
    c.l1 = __fsub_rn(s, (float)c.i0);
    c.l0 = __fsub_rn(1.0f, c.l1);
    return c;
}

// h0*(w0*v00 + w1*v01) + h1*(w0*v10 + w1*v11), contracted as nvcc contracts ATen's expression
__device__ __forceinline__ void blend_up(const UpCoef &cy, const UpCoef &cx, float x00, float y00, float x01, float y01,
                                         float x10, float y10, float x11, float y11, float &gx, float &gy)
{
    gx = __fmaf_rn(cy.l0, __fmaf_rn(cx.l0, x00, __fmul_rn(cx.l1, x01)), __fmul_rn(cy.l1, __fmaf_rn(cx.l0, x10, __fmul_rn(cx.l1, x11))));
    gy = __fmaf_rn(cy.l0, __fmaf_rn(cx.l0, y00, __fmul_rn(cx.l1, y01)), __fmul_rn(cy.l1, __fmaf_rn(cx.l0, y10, __fmul_rn(cx.l1, y11))));
}

// the upsampled map from the row / column coefficients of an output pixel
template <typename L>
__device__ __forceinline__ void map_up(const MapSpec &m, int n, const UpCoef &cy, const UpCoef &cx, float &gx, float &gy)
{
    float x00, y00, x01, y01, x10, y10, x11, y11;
    lattice_map<L>(m, n, cy.i0, cx.i0, x00, y00);
    lattice_map<L>(m, n, cy.i0, cx.i0 + cx.ip, x01, y01);
    lattice_map<L>(m, n, cy.i0 + cy.ip, cx.i0, x10, y10);
    lattice_map<L>(m, n, cy.i0 + cy.ip, cx.i0 + cx.ip, x11, y11);
    blend_up(cy, cx, x00, y00, x01, y01, x10, y10, x11, y11, gx, gy);
}

// the map the sampler sees at output pixel (h, w)
template <typename L>
__device__ __forceinline__ void map_at(const MapSpec &m, int n, int h, int w, float rh, float rw, float &gx, float &gy)
{
    if (m.upsample == PWS_UP_NONE) { lattice_map<L>(m, n, h, w, gx, gy); return; }
    const bool al = m.upsample == PWS_UP_ALIGNED;
    map_up<L>(m, n, up_coef(h, m.mh, rh, al), up_coef(w, m.mw, rw, al), gx, gy);
}

__device__ __forceinline__ void up_scales(const MapSpec &m, int Ho, int Wo, float &rh, float &rw)
{
    rh = rw = 0.f;
    if (m.upsample == PWS_UP_ALIGNED) {
        rh = Ho > 1 ? __fdiv_rn((float)(m.mh - 1), (float)(Ho - 1)) : 0.f;
        rw = Wo > 1 ? __fdiv_rn((float)(m.mw - 1), (float)(Wo - 1)) : 0.f;
    } else if (m.upsample == PWS_UP_HALF_PIXEL) {
        rh = __fdiv_rn((float)m.mh, (float)Ho);
        rw = __fdiv_rn((float)m.mw, (float)Wo);
    }
}

// host twin (float division is correctly rounded on both sides)
inline void up_scales_host(const MapSpec &m, int Ho, int Wo, float &rh, float &rw)
{
    rh = rw = 0.f;
    if (m.upsample == PWS_UP_ALIGNED) {
        rh = Ho > 1 ? (float)(m.mh - 1) / (float)(Ho - 1) : 0.f;
        rw = Wo > 1 ? (float)(m.mw - 1) / (float)(Wo - 1) : 0.f;
    } else if (m.upsample == PWS_UP_HALF_PIXEL) {
        rh = (float)m.mh / (float)Ho;
        rw = (float)m.mw / (float)Wo;
    }
}

template <typename T> __device__ __forceinline__ float load_px(const T *p) { return to_acc(ldg(p)); }
template <> __device__ __forceinline__ float load_px<uint8_t>(const uint8_t *p) { return (float)__ldg(p); }
template <typename T> __device__ __forceinline__ void store_px(T *p, float v) { *p = from_acc<T, float>(v); }
// uint8 egress: truncation, what `.astype(np.uint8)` does to the in-range values a warp of 0..255 produces
template <> __device__ __forceinline__ void store_px<uint8_t>(uint8_t *p, float v) { *p = (uint8_t)(int)fminf(fmaxf(v, 0.f), 255.f); }

constexpr int kTileW = 64, kTileH = 16, kThreads = 256;

// a lattice node read as one vector, upcast (exact)
__device__ __forceinline__ float2 node_f2(float2 v) { return v; }
__device__ __forceinline__ float2 node_f2(__half2 v) { return __half22float2(v); }
__device__ __forceinline__ float2 node_f2(__nv_bfloat162 v) { return __bfloat1622float2(v); }

template <typename TI, typename TO, typename L, int CS>
__global__ void __launch_bounds__(kThreads)
fwd_fused_kernel(const View in, const MapSpec m, const View out, const Geometry g)
{
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int n = blockIdx.z;
    const TI *__restrict__ ip = (const TI *)in.p + (int64_t)n * in.sN;
    TO *__restrict__ op = (TO *)out.p + (int64_t)n * out.sN;
    const bool align = g.align != 0;
    const int C = CS > 0 ? CS : g.C;
    float rh, rw;
    up_scales(m, g.Ho, g.Wo, rh, rw);

    float gx[2][2], gy[2][2];
    if (m.upsample == PWS_UP_NONE) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
                gx[j][i] = 0.f; gy[j][i] = 0.f;
                if (w < g.Wo && h < g.Ho) lattice_map<L>(m, n, h, w, gx[j][i], gy[j][i]);
            }
    } else {
        // a thread's four pixels share two rows and two columns: two row and two column coefficient sets
        const bool al = m.upsample == PWS_UP_ALIGNED;
        UpCoef cy[2], cx[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) cy[j] = up_coef(min(blockIdx.y * kTileH + wrp + 8 * j, g.Ho - 1), m.mh, rh, al);
#pragma unroll
        for (int i = 0; i < 2; ++i) cx[i] = up_coef(min(blockIdx.x * kTileW + lane + 32 * i, g.Wo - 1), m.mw, rw, al);
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int i = 0; i < 2; ++i) map_up<L>(m, n, cy[j], cx[i], gx[j][i], gy[j][i]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
            if (!(w < g.Wo && h < g.Ho)) continue;
            Taps<float> t;
            make_taps(source_index(gx[j][i], g.W, g.padding, align), source_index(gy[j][i], g.H, g.padding, align), g.H, g.W, t);
            const int o_nw = t.y0 * in.s2 + t.x0 * in.s3;
            const int o_out = h * out.s2 + w * out.s3;
#pragma unroll 3
            for (int c = 0; c < C; ++c) {
                const TI *__restrict__ pc = ip + c * in.s1;
                float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
                if (t.mask & 1u) v0 = load_px(pc + o_nw);
                if (t.mask & 2u) v1 = load_px(pc + o_nw + in.s3);
                if (t.mask & 4u) v2 = load_px(pc + o_nw + in.s2);
                if (t.mask & 8u) v3 = load_px(pc + o_nw + in.s2 + in.s3);
                if (m.has_pre) {  // (x + a) * b, elementwise as the reference does before sampling
                    v0 = __fmul_rn(__fadd_rn(v0, m.pre_add), m.pre_mul); v1 = __fmul_rn(__fadd_rn(v1, m.pre_add), m.pre_mul);
                    v2 = __fmul_rn(__fadd_rn(v2, m.pre_add), m.pre_mul); v3 = __fmul_rn(__fadd_rn(v3, m.pre_add), m.pre_mul);
                }
                float acc = 0.f;
                if (t.mask & 1u) acc = ffma(v0, t.nw, acc);
                if (t.mask & 2u) acc = ffma(v1, t.ne, acc);
                if (t.mask & 4u) acc = ffma(v2, t.sw, acc);
                if (t.mask & 8u) acc = ffma(v3, t.se, acc);
                if (m.has_post) acc = __fadd_rn(__fdiv_rn(acc, m.post_div), m.post_add);
                store_px(op + o_out + c * out.s1, acc);
            }
        }
}

// The inference site, specialised (R/main_new.py:679-684,697-721): uint8 HWC frame in, uint8 HWC frame out, the map
// is the bilinear upsample of a dense interleaved low-resolution lattice (what the host side composes once per call).
// Same arithmetic as the generic kernel above, statement for statement -- only the addressing is compile-time: the
// generic kernel spends 390 instructions per pixel, most of them on run-time strides and layout checks, and is
// issue-bound (79 % of the issue slots).  LP: one lattice node, float2 or the __half2 / __nv_bfloat162 of a 16-bit lattice.
// Without a minimum-blocks hint ptxas caps the kUpAligned instantiations at 32 registers and spills 8 bytes; the 16-bit
// ones ask for one block per SM and get 66-72 registers, no spill (the fp32 ones keep the code they have always had).
template <typename LP> constexpr int kU8MinBlocks = sizeof(LP) == 8 ? 0 : 1;
template <typename LP, bool kBorder, bool kAlignCorners, bool kUpAligned>
__global__ void __launch_bounds__(kThreads, kU8MinBlocks<LP>)
fwd_fused_u8_kernel(const uint8_t *__restrict__ in, const LP *__restrict__ lattice, uint8_t *__restrict__ out,
                    const int H, const int W, const int Ho, const int Wo, const int mh, const int mw, const float rh, const float rw)
{
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int n = blockIdx.z;
    const uint8_t *__restrict__ ip = in + (int64_t)n * H * W * 3;
    uint8_t *__restrict__ op = out + (int64_t)n * Ho * Wo * 3;
    const LP *__restrict__ L = lattice + (int64_t)n * mh * mw;
    const int padding = kBorder ? PWS_PAD_BORDER : PWS_PAD_ZEROS;

    UpCoef cy[2], cx[2];
    int hh[2], ww[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) { hh[j] = blockIdx.y * kTileH + wrp + 8 * j; cy[j] = up_coef(min(hh[j], Ho - 1), mh, rh, kUpAligned); }
#pragma unroll
    for (int i = 0; i < 2; ++i) { ww[i] = blockIdx.x * kTileW + lane + 32 * i; cx[i] = up_coef(min(ww[i], Wo - 1), mw, rw, kUpAligned); }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            if (!(ww[i] < Wo && hh[j] < Ho)) continue;
            const LP *r0 = L + cy[j].i0 * mw + cx[i].i0, *r1 = r0 + cy[j].ip * mw;
            const float2 v00 = node_f2(__ldg(r0)), v01 = node_f2(__ldg(r0 + cx[i].ip)), v10 = node_f2(__ldg(r1)), v11 = node_f2(__ldg(r1 + cx[i].ip));
            // h0*(w0*v00 + w1*v01) + h1*(w0*v10 + w1*v11), contracted as in map_up()
            const float gx = __fmaf_rn(cy[j].l0, __fmaf_rn(cx[i].l0, v00.x, __fmul_rn(cx[i].l1, v01.x)), __fmul_rn(cy[j].l1, __fmaf_rn(cx[i].l0, v10.x, __fmul_rn(cx[i].l1, v11.x))));
            const float gy = __fmaf_rn(cy[j].l0, __fmaf_rn(cx[i].l0, v00.y, __fmul_rn(cx[i].l1, v01.y)), __fmul_rn(cy[j].l1, __fmaf_rn(cx[i].l0, v10.y, __fmul_rn(cx[i].l1, v11.y))));
            Taps<float> t;
            make_taps(source_index(gx, W, padding, kAlignCorners), source_index(gy, H, padding, kAlignCorners), H, W, t);
            const uint8_t *__restrict__ p0 = ip + ((int64_t)t.y0 * W + t.x0) * 3;
            const uint8_t *__restrict__ p1 = p0 + W * 3;
            uint8_t *__restrict__ o = op + ((int64_t)hh[j] * Wo + ww[i]) * 3;
            if (t.mask == 15u) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    float acc = ffma((float)__ldg(p0 + c), t.nw, 0.f);
                    acc = ffma((float)__ldg(p0 + 3 + c), t.ne, acc);
                    acc = ffma((float)__ldg(p1 + c), t.sw, acc);
                    acc = ffma((float)__ldg(p1 + 3 + c), t.se, acc);
                    store_px(o + c, acc);
                }
            } else {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    float acc = 0.f;
                    if (t.mask & 1u) acc = ffma((float)__ldg(p0 + c), t.nw, acc);
                    if (t.mask & 2u) acc = ffma((float)__ldg(p0 + 3 + c), t.ne, acc);
                    if (t.mask & 4u) acc = ffma((float)__ldg(p1 + c), t.sw, acc);
                    if (t.mask & 8u) acc = ffma((float)__ldg(p1 + 3 + c), t.se, acc);
                    store_px(o + c, acc);
                }
            }
        }
}

template <typename L>
__global__ void __launch_bounds__(256)
compose_map_kernel(const MapSpec m, const View out, const int N, const int Ho, const int Wo)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)N * Ho * Wo) return;
    const int w = (int)(idx % Wo);
    const int64_t r = idx / Wo;
    const int h = (int)(r % Ho), n = (int)(r / Ho);
    float rh, rw, gx, gy;
    up_scales(m, Ho, Wo, rh, rw);
    map_at<L>(m, n, h, w, rh, rw, gx, gy);
    float *o = (float *)out.p + (int64_t)n * out.sN + h * out.s1 + w * out.s2;
    o[0] = gx; o[out.s3] = gy;
}

// ---- backward ----------------------------------------------------------------------------------------------------
// grad_output of a differentiable fused call: fp32 for fp32 and uint8 frames, the frame's type for 16-bit frames
template <typename T> struct GradOut { using type = T; };
template <> struct GradOut<uint8_t> { using type = float; };

// lattice nodes one backward CTA composes into shared memory (10 KB): an upsample (lattice no finer than the output) spans
// at most 17 x 65 nodes per 64 x 16 tile
constexpr int kWinNodes = 1280;

// Autograd of fwd_fused_kernel.  Per output pixel: the map with the forward's statements (same taps), go = gout / d (the
// forward's true division), grad_grid in ATen's statement order on the pre-scaled taps (as stages_bwd_kernel), optional
// grad_input REDs, and d loss / d lattice:
//   no upsample: the pixel is its lattice node, a plain store;
//   upsample:    the pair goes to the four nodes map_up() read, with its weights.  The 32 lanes of a warp row share the row
//                coefficients and cx.i0 is non-decreasing across them, so pixels of one lattice column form a run of lanes:
//                a segmented shuffle scan sums each run and its last lane issues one 8-byte RED per node.  At 1080p
//                from 256^2 a warp row spans ~5 columns: ~20 REDs instead of 256.  (A lattice finer than the output
//                gives runs of one lane: correct, not tuned.)  Shared-memory float atomics are CAS loops on sm_100a.
// Without a minimum-blocks hint ptxas caps some instantiations at 64 registers and spills; two blocks per SM (up to 128
// registers) lets every instantiation keep its 60-96 without spilling.
template <typename TI, typename L, int CS, bool kGin>
__global__ void __launch_bounds__(kThreads, 2)
bwd_fused_kernel(const View gout, const View in, const MapSpec m, const View gin, float *__restrict__ glat, const Geometry g)
{
    using TG = typename GradOut<TI>::type;
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int n = blockIdx.z;
    const TI *__restrict__ ip = (const TI *)in.p + (int64_t)n * in.sN;
    const TG *__restrict__ gop = (const TG *)gout.p + (int64_t)n * gout.sN;
    float *__restrict__ gip = kGin ? (float *)gin.p + (int64_t)n * gin.sN : nullptr;
    float *__restrict__ glp = glat ? glat + (int64_t)n * m.mh * m.mw * 2 : nullptr;
    const bool align = g.align != 0, up = m.upsample != PWS_UP_NONE;
    const int C = CS > 0 ? CS : g.C;
    float rh, rw;
    up_scales(m, g.Ho, g.Wo, rh, rw);

    float gx[2][2], gy[2][2];
    UpCoef cy[2], cx[2];
    if (!up) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
                gx[j][i] = 0.f; gy[j][i] = 0.f;
                if (w < g.Wo && h < g.Ho) lattice_map<L>(m, n, h, w, gx[j][i], gy[j][i]);
            }
    } else {
        const bool al = m.upsample == PWS_UP_ALIGNED;
#pragma unroll
        for (int j = 0; j < 2; ++j) cy[j] = up_coef(min(blockIdx.y * kTileH + wrp + 8 * j, g.Ho - 1), m.mh, rh, al);
#pragma unroll
        for (int i = 0; i < 2; ++i) cx[i] = up_coef(min(blockIdx.x * kTileW + lane + 32 * i, g.Wo - 1), m.mw, rw, al);
        // The tile's lattice nodes, composed once per CTA into shared memory: up_coef is monotone in the output index, so
        // every node the tile's pixels blend lies in the window spanned by its first and last row and column.  Upsampling
        // evaluates four nodes per pixel, and a node with a base costs IEEE divisions and a planar drift two scalar loads;
        // at 1080p from 256^2 a tile needs ~66 nodes where its pixels would evaluate 4096.  The values are lattice_map's,
        // so the map is the forward's bit for bit.  A lattice much finer than the output (a downsample) overflows the
        // window and evaluates per pixel.
        const UpCoef t0 = up_coef(blockIdx.y * kTileH, m.mh, rh, al), t1 = up_coef(min(blockIdx.y * kTileH + kTileH - 1, g.Ho - 1), m.mh, rh, al);
        const UpCoef s0 = up_coef(blockIdx.x * kTileW, m.mw, rw, al), s1 = up_coef(min(blockIdx.x * kTileW + kTileW - 1, g.Wo - 1), m.mw, rw, al);
        const int nr = t1.i0 + t1.ip - t0.i0 + 1, nc = s1.i0 + s1.ip - s0.i0 + 1;
        if ((int64_t)nr * nc <= kWinNodes) {   // uniform across the CTA
            __shared__ float2 win[kWinNodes];
            for (int k = threadIdx.x; k < nr * nc; k += kThreads) {
                float x, y;
                lattice_map<L>(m, n, t0.i0 + k / nc, s0.i0 + k % nc, x, y);
                win[k] = make_float2(x, y);
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const float2 *r0 = win + (cy[j].i0 - t0.i0) * nc + (cx[i].i0 - s0.i0), *r1 = r0 + cy[j].ip * nc;
                    const float2 v00 = r0[0], v01 = r0[cx[i].ip], v10 = r1[0], v11 = r1[cx[i].ip];
                    blend_up(cy[j], cx[i], v00.x, v00.y, v01.x, v01.y, v10.x, v10.y, v11.x, v11.y, gx[j][i], gy[j][i]);
                }
        } else {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int i = 0; i < 2; ++i) map_up<L>(m, n, cy[j], cx[i], gx[j][i], gy[j][i]);
        }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int w = blockIdx.x * kTileW + lane + 32 * i, h = blockIdx.y * kTileH + wrp + 8 * j;
            const bool valid = w < g.Wo && h < g.Ho;
            float px = 0.f, py = 0.f;   // d loss / d map at (h, w)
            if (valid) {
                float gxm, gym;
                const float ix = source_index_set_grad(gx[j][i], g.W, g.padding, align, &gxm);
                const float iy = source_index_set_grad(gy[j][i], g.H, g.padding, align, &gym);
                Taps<float> t;
                make_taps(ix, iy, g.H, g.W, t);
                const float x0f = (float)t.x0, y0f = (float)t.y0;
                const float dw = fsub(x0f + 1.0f, ix), de = fsub(ix, x0f), dn = fsub(y0f + 1.0f, iy), ds = fsub(iy, y0f);
                const int o_nw = t.y0 * in.s2 + t.x0 * in.s3;
                const int o_go = h * gout.s2 + w * gout.s3;
                float gix = 0.f, giy = 0.f;
#pragma unroll 3
                for (int c = 0; c < C; ++c) {
                    float go = to_acc(ldg(gop + o_go + c * gout.s1));
                    if (m.has_post) go = __fdiv_rn(go, m.post_div);   // d (acc / d + e) / d acc, as the forward divides
                    if (glp) {
                        const TI *__restrict__ pc = ip + c * in.s1;
                        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
                        if (t.mask & 1u) v0 = load_px(pc + o_nw);
                        if (t.mask & 2u) v1 = load_px(pc + o_nw + in.s3);
                        if (t.mask & 4u) v2 = load_px(pc + o_nw + in.s2);
                        if (t.mask & 8u) v3 = load_px(pc + o_nw + in.s2 + in.s3);
                        if (m.has_pre) {
                            v0 = __fmul_rn(__fadd_rn(v0, m.pre_add), m.pre_mul); v1 = __fmul_rn(__fadd_rn(v1, m.pre_add), m.pre_mul);
                            v2 = __fmul_rn(__fadd_rn(v2, m.pre_add), m.pre_mul); v3 = __fmul_rn(__fadd_rn(v3, m.pre_add), m.pre_mul);
                        }
                        // ATen's statement order: t = v*d rounded, then one fma with gOut
                        if (t.mask & 1u) { gix = ffma(-fmul(v0, dn), go, gix); giy = ffma(-fmul(v0, dw), go, giy); }
                        if (t.mask & 2u) { gix = ffma(fmul(v1, dn), go, gix);  giy = ffma(-fmul(v1, de), go, giy); }
                        if (t.mask & 4u) { gix = ffma(-fmul(v2, ds), go, gix); giy = ffma(fmul(v2, dw), go, giy); }
                        if (t.mask & 8u) { gix = ffma(fmul(v3, ds), go, gix);  giy = ffma(fmul(v3, de), go, giy); }
                    }
                    if (kGin) {   // d out / d frame = w_tap, through the pre scale (x + a) * b: times b
                        const float gs = m.has_pre ? __fmul_rn(go, m.pre_mul) : go;
                        float *pg = gip + c * gin.s1 + t.y0 * gin.s2 + t.x0;
                        if (t.mask & 1u) atomicAdd(pg, fmul(t.nw, gs));
                        if (t.mask & 2u) atomicAdd(pg + 1, fmul(t.ne, gs));
                        if (t.mask & 4u) atomicAdd(pg + gin.s2, fmul(t.sw, gs));
                        if (t.mask & 8u) atomicAdd(pg + gin.s2 + 1, fmul(t.se, gs));
                    }
                }
                px = fmul(gxm, gix); py = fmul(gym, giy);
            }
            if (!glp) continue;
            if (!up) {
                if (valid) st_pair(glp + ((int64_t)h * m.mw + w) * 2, px, py);
                continue;
            }
            if (h >= g.Ho) continue;   // a warp row shares h: uniform across the shuffles below
            // column sums of the run: node column i0 takes l0 * pair, column i0 + ip takes l1 * pair (lanes past the
            // right edge carry zeros and the clamped column, so they join the last run)
            const int key = cx[i].i0;
            float a0 = fmul(cx[i].l0, px), a1 = fmul(cx[i].l0, py), b0 = fmul(cx[i].l1, px), b1 = fmul(cx[i].l1, py);
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int k = __shfl_up_sync(0xffffffffu, key, d);
                const float ta0 = __shfl_up_sync(0xffffffffu, a0, d), ta1 = __shfl_up_sync(0xffffffffu, a1, d);
                const float tb0 = __shfl_up_sync(0xffffffffu, b0, d), tb1 = __shfl_up_sync(0xffffffffu, b1, d);
                if (lane >= d && k == key) { a0 = __fadd_rn(a0, ta0); a1 = __fadd_rn(a1, ta1); b0 = __fadd_rn(b0, tb0); b1 = __fadd_rn(b1, tb1); }
            }
            const int knext = __shfl_down_sync(0xffffffffu, key, 1);
            if (lane == 31 || knext != key) {
                float *r0 = glp + ((int64_t)cy[j].i0 * m.mw + key) * 2;
                float *r1 = r0 + (int64_t)cy[j].ip * m.mw * 2;
                const int dc = cx[i].ip * 2;
                const float h0 = cy[j].l0, h1 = cy[j].l1;
                // one 8-byte vector RED per node (glattice is 8-byte aligned, checked in capi.cu)
                atomicAdd(reinterpret_cast<float2 *>(r0), make_float2(fmul(h0, a0), fmul(h0, a1)));
                atomicAdd(reinterpret_cast<float2 *>(r0 + dc), make_float2(fmul(h0, b0), fmul(h0, b1)));
                atomicAdd(reinterpret_cast<float2 *>(r1), make_float2(fmul(h1, a0), fmul(h1, a1)));
                atomicAdd(reinterpret_cast<float2 *>(r1 + dc), make_float2(fmul(h1, b0), fmul(h1, b1)));
            }
        }
}

// d loss / d theta of the affine base: gtheta[n, c, :] = sum_ij glattice[n, i, j, c] * (bx_j, by_i, 1), one block per item,
// fixed summation order (strided per thread, then a tree), so the result does not depend on the REDs' order beyond glattice
constexpr int kThetaThreads = 256;
__global__ void __launch_bounds__(kThetaThreads)
theta_grad_kernel(const float *__restrict__ glat, const MapSpec m, float *__restrict__ gtheta)
{
    const int n = blockIdx.x;
    const float *__restrict__ gl = glat + (int64_t)n * m.mh * m.mw * 2;
    float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int64_t nodes = (int64_t)m.mh * m.mw;
    for (int64_t k = threadIdx.x; k < nodes; k += kThetaThreads) {
        const int i = (int)(k / m.mw), j = (int)(k % m.mw);
        const float bx = lattice_base(j, m.mw, m.base, m.base_align), by = lattice_base(i, m.mh, m.base, m.base_align);
        const float2 v = *reinterpret_cast<const float2 *>(gl + 2 * k);
        s[0] = __fmaf_rn(v.x, bx, s[0]); s[1] = __fmaf_rn(v.x, by, s[1]); s[2] = __fadd_rn(v.x, s[2]);
        s[3] = __fmaf_rn(v.y, bx, s[3]); s[4] = __fmaf_rn(v.y, by, s[4]); s[5] = __fadd_rn(v.y, s[5]);
    }
    __shared__ float red[6][kThetaThreads];
#pragma unroll
    for (int q = 0; q < 6; ++q) red[q][threadIdx.x] = s[q];
    __syncthreads();
    for (int half = kThetaThreads / 2; half > 0; half >>= 1) {
        if (threadIdx.x < half)
#pragma unroll
            for (int q = 0; q < 6; ++q) red[q][threadIdx.x] = __fadd_rn(red[q][threadIdx.x], red[q][threadIdx.x + half]);
        __syncthreads();
    }
    if (threadIdx.x < 6) gtheta[n * 6 + threadIdx.x] = red[threadIdx.x][0];
}

template <typename TI, typename L>
void launch_bwd_l(const View &gout, const View &in, const MapSpec &m, const View &gin, bool want_gin, float *glat,
                  const Geometry &g, cudaStream_t st)
{
    dim3 blocks((g.Wo + kTileW - 1) / kTileW, (g.Ho + kTileH - 1) / kTileH, g.N);
#define PWS_BF(CS, GIN) bwd_fused_kernel<TI, L, CS, GIN><<<blocks, kThreads, 0, st>>>(gout, in, m, gin, glat, g)
    if constexpr (!std::is_same<TI, uint8_t>::value) {   // a uint8 frame has no gradient
        if (want_gin) {
            if (g.C == 3) PWS_BF(3, true); else if (g.C == 1) PWS_BF(1, true); else PWS_BF(0, true);
            return;
        }
    }
    if (g.C == 3) PWS_BF(3, false); else if (g.C == 1) PWS_BF(1, false); else PWS_BF(0, false);
#undef PWS_BF
}

template <typename TI>
void launch_bwd(const View &gout, const View &in, const MapSpec &m, const View &gin, bool want_gin, float *glat,
                const Geometry &g, cudaStream_t st)
{
    if (m.drift_dtype == PWS_F16) launch_bwd_l<TI, __half>(gout, in, m, gin, want_gin, glat, g, st);
    else if (m.drift_dtype == PWS_BF16) launch_bwd_l<TI, __nv_bfloat16>(gout, in, m, gin, want_gin, glat, g, st);
    else launch_bwd_l<TI, float>(gout, in, m, gin, want_gin, glat, g, st);
}

template <typename TI, typename TO, typename L>
void launch_io_l(const View &in, const MapSpec &m, const View &out, const Geometry &g, cudaStream_t st)
{
    dim3 blocks((g.Wo + kTileW - 1) / kTileW, (g.Ho + kTileH - 1) / kTileH, g.N);
    if (g.C == 3) { fwd_fused_kernel<TI, TO, L, 3><<<blocks, kThreads, 0, st>>>(in, m, out, g); note_launch(); }
    else if (g.C == 1) { fwd_fused_kernel<TI, TO, L, 1><<<blocks, kThreads, 0, st>>>(in, m, out, g); note_launch(); }
    else { fwd_fused_kernel<TI, TO, L, 0><<<blocks, kThreads, 0, st>>>(in, m, out, g); note_launch(); }
    note_kernel("fwd_fused");
}

template <typename TI, typename TO>
void launch_io(const View &in, const MapSpec &m, const View &out, const Geometry &g, cudaStream_t st)
{
    if (m.drift_dtype == PWS_F16) launch_io_l<TI, TO, __half>(in, m, out, g, st);
    else if (m.drift_dtype == PWS_BF16) launch_io_l<TI, TO, __nv_bfloat16>(in, m, out, g, st);
    else launch_io_l<TI, TO, float>(in, m, out, g, st);
}

template <typename LP>
void launch_u8(const View &in, const MapSpec &m, const View &out, const Geometry &g, cudaStream_t st)
{
    dim3 blocks((g.Wo + kTileW - 1) / kTileW, (g.Ho + kTileH - 1) / kTileH, g.N);
    float rh, rw;
    up_scales_host(m, g.Ho, g.Wo, rh, rw);
    const uint8_t *ip = (const uint8_t *)in.p;
    const LP *lp = (const LP *)m.drift.p;
    uint8_t *op = (uint8_t *)out.p;
    const bool border = g.padding == PWS_PAD_BORDER, al = g.align != 0, upa = m.upsample == PWS_UP_ALIGNED;
#define PWS_U8(B, A, U) fwd_fused_u8_kernel<LP, B, A, U><<<blocks, kThreads, 0, st>>>(ip, lp, op, g.H, g.W, g.Ho, g.Wo, m.mh, m.mw, rh, rw)
    if (border) { if (al) { if (upa) PWS_U8(true, true, true); else PWS_U8(true, true, false); } else { if (upa) PWS_U8(true, false, true); else PWS_U8(true, false, false); } }
    else        { if (al) { if (upa) PWS_U8(false, true, true); else PWS_U8(false, true, false); } else { if (upa) PWS_U8(false, false, true); else PWS_U8(false, false, false); } }
#undef PWS_U8
}

}  // namespace

int launch_forward_fused(const View &in, int in_dtype, const MapSpec &m, const View &out, int out_dtype,
                         const Geometry &g, cudaStream_t st)
{
    if (g.N > 65535 || (g.Ho + kTileH - 1) / kTileH > 65535) { set_error("fused forward: batch or height too large"); return PWS_EUNSUPPORTED; }
    // the inference site: dense uint8 HWC in and out, dense interleaved lattice (fp32 or 16-bit), upsampling, nothing else
    const int lat_bytes = m.drift_dtype == PWS_F32 ? 4 : 2;
    const bool u8_fast = in_dtype == PWS_U8 && out_dtype == PWS_U8 && g.C == 3 && m.base == PWS_BASE_NONE && m.drift.p &&
        m.upsample != PWS_UP_NONE && !m.has_pre && !m.has_post &&
        in.s1 == 1 && in.s3 == 3 && in.s2 == 3 * g.W && (g.N == 1 || in.sN == (int64_t)3 * g.W * g.H) &&
        out.s1 == 1 && out.s3 == 3 && out.s2 == 3 * g.Wo && (g.N == 1 || out.sN == (int64_t)3 * g.Wo * g.Ho) &&
        m.drift.s3 == 1 && m.drift.s2 == 2 && m.drift.s1 == 2 * m.mw && (g.N == 1 || m.drift.sN == (int64_t)2 * m.mw * m.mh) &&
        !(reinterpret_cast<uintptr_t>(m.drift.p) & (2 * lat_bytes - 1));
    if (u8_fast) {
        if (m.drift_dtype == PWS_F16) launch_u8<__half2>(in, m, out, g, st);
        else if (m.drift_dtype == PWS_BF16) launch_u8<__nv_bfloat162>(in, m, out, g, st);
        else launch_u8<float2>(in, m, out, g, st);
        note_launch();
        note_kernel("fwd_fused_u8");
        return PWS_OK;
    }
    if (in_dtype == PWS_F32 && out_dtype == PWS_F32) launch_io<float, float>(in, m, out, g, st);
    else if (in_dtype == PWS_U8 && out_dtype == PWS_F32) launch_io<uint8_t, float>(in, m, out, g, st);
    else if (in_dtype == PWS_U8 && out_dtype == PWS_U8) launch_io<uint8_t, uint8_t>(in, m, out, g, st);
    else if (in_dtype == PWS_F32 && out_dtype == PWS_U8) launch_io<float, uint8_t>(in, m, out, g, st);
    else if (in_dtype == PWS_BF16 && out_dtype == PWS_BF16) launch_io<__nv_bfloat16, __nv_bfloat16>(in, m, out, g, st);
    else if (in_dtype == PWS_F16 && out_dtype == PWS_F16) launch_io<__half, __half>(in, m, out, g, st);
    else { set_error("fused forward: unsupported frame/output dtype pair (%d -> %d)", in_dtype, out_dtype); return PWS_EUNSUPPORTED; }
    return PWS_OK;
}

int launch_compose_map(const MapSpec &m, const View &out, int N, int Ho, int Wo, cudaStream_t st)
{
    const int64_t total = (int64_t)N * Ho * Wo;
    if (total == 0) return PWS_OK;
    const int64_t blocks = (total + 255) / 256;
    if (blocks > INT_MAX) { set_error("compose_map: too many pixels"); return PWS_EUNSUPPORTED; }
    if (m.drift_dtype == PWS_F16) compose_map_kernel<__half><<<(unsigned)blocks, 256, 0, st>>>(m, out, N, Ho, Wo);
    else if (m.drift_dtype == PWS_BF16) compose_map_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>(m, out, N, Ho, Wo);
    else compose_map_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(m, out, N, Ho, Wo);
    note_launch();
    note_kernel("compose_map");
    return PWS_OK;
}

int launch_backward_fused(const View &gout, const View &in, int in_dtype, const MapSpec &m, const View &gin, bool want_gin,
                          float *glat, float *gtheta, const Geometry &g, cudaStream_t st)
{
    if (g.N > 65535 || (g.Ho + kTileH - 1) / kTileH > 65535) { set_error("fused backward: batch or height too large"); return PWS_EUNSUPPORTED; }
    if (want_gin) {
        cudaError_t e = cudaMemsetAsync(gin.p, 0, (size_t)g.N * g.C * g.H * g.W * sizeof(float), st);
        if (e != cudaSuccess) { set_error("fused backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
    }
    if (glat && m.upsample != PWS_UP_NONE) {   // the upsample's adjoint accumulates; without it every node is stored once
        cudaError_t e = cudaMemsetAsync(glat, 0, (size_t)g.N * m.mh * m.mw * 2 * sizeof(float), st);
        if (e != cudaSuccess) { set_error("fused backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
    }
    if (!want_gin && !glat) return PWS_OK;
    if (in_dtype == PWS_F32) launch_bwd<float>(gout, in, m, gin, want_gin, glat, g, st);
    else if (in_dtype == PWS_U8) launch_bwd<uint8_t>(gout, in, m, gin, false, glat, g, st);
    else if (in_dtype == PWS_F16) launch_bwd<__half>(gout, in, m, gin, want_gin, glat, g, st);
    else if (in_dtype == PWS_BF16) launch_bwd<__nv_bfloat16>(gout, in, m, gin, want_gin, glat, g, st);
    else { set_error("fused backward: unsupported frame dtype %d", in_dtype); return PWS_EUNSUPPORTED; }
    note_launch();
    if (gtheta) { theta_grad_kernel<<<g.N, kThetaThreads, 0, st>>>(glat, m, gtheta); note_launch(); }
    note_kernel("bwd_fused");
    return PWS_OK;
}

}  // namespace pws
