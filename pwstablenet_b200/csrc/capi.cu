// capi.cu -- extern "C" boundary of libpwswarp.so (include/pwswarp.h).
// Validation mirrors check_grid_sampler_common / check_grid_sampler_2d
// ($TORCH/include/ATen/native/GridSamplerUtils.h:23-71); messages keep ATen's
// "grid_sampler(): ..." wording so the Python shim can re-raise them verbatim.
#include "pws_common.cuh"

#include <atomic>
#include <cstdarg>
#include <cstdio>

namespace pws {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static thread_local const char *g_last_kernel = "";
static std::atomic<int64_t> g_small_elems{(int64_t)PWS_SMALL_ELEMS};
int64_t small_problem_threshold() { return g_small_elems.load(std::memory_order_relaxed); }
void note_launch(int kernels) { g_launches.fetch_add((uint64_t)kernels, std::memory_order_relaxed); }
void note_kernel(const char *family) { g_last_kernel = family; }

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define PWS_TRY(expr) do { int rc_ = (expr); if (rc_ != PWS_OK) return rc_; } while (0)

namespace {

int elem_size(int dt)
{
    switch (dt) {
        case PWS_F32: return 4;
        case PWS_F16: case PWS_BF16: return 2;
        case PWS_F64: return 8;
        case PWS_U8: return 1;
        case PWS_I32: return 4;
        default: return 0;
    }
}

// extent (in elements) one batch item of `t` spans, over dims 1..3
int64_t item_span(const pws_tensor *t)
{
    int64_t s = 1;
    for (int d = 1; d < 4; ++d) {
        if (t->size[d] == 0) return 0;
        const int64_t st = t->stride[d] < 0 ? -t->stride[d] : t->stride[d];
        s += (t->size[d] - 1) * st;
    }
    return s;
}

const char *dtype_name(int dt)
{
    static const char *const names[] = {"f32", "f16", "bf16", "f64", "u8", "i32"};
    return elem_size(dt) ? names[dt] : "?";
}

// set_error with the argument's name in front: "grad_grid: ..." or, for stage k's tensors, "grad_grid 1: ..."
int arg_error(int rc, const char *what, int k, const char *fmt, ...)
{
    int n = k < 0 ? snprintf(g_err, sizeof(g_err), "%s: ", what) : snprintf(g_err, sizeof(g_err), "%s %d: ", what, k);
    if (n < 0 || n >= (int)sizeof(g_err)) n = 0;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err + n, sizeof(g_err) - n, fmt, ap);
    va_end(ap);
    return rc;
}

int make_view(const pws_tensor *t, const char *what, int k, View *v)
{
    if (!t) return arg_error(PWS_EINVAL, what, k, "null tensor descriptor");
    if (elem_size(t->dtype) == 0) return arg_error(PWS_EINVAL, what, k, "unknown dtype %d", t->dtype);
    for (int d = 0; d < 4; ++d) {
        if (t->size[d] < 0) return arg_error(PWS_EINVAL, what, k, "negative size");
        if (t->stride[d] < 0) return arg_error(PWS_EUNSUPPORTED, what, k, "negative strides are not supported");
        if (t->size[d] > INT_MAX) return arg_error(PWS_EUNSUPPORTED, what, k, "dimension %d too large", d);
    }
    if (item_span(t) >= ((int64_t)1 << 31))
        return arg_error(PWS_EUNSUPPORTED, what, k, "one batch item spans >= 2^31 elements (32-bit in-frame offsets)");
    const int64_t numel = t->size[0] * t->size[1] * t->size[2] * t->size[3];
    if (numel > 0 && !t->data) return arg_error(PWS_EINVAL, what, k, "null data pointer");
    v->p = t->data;
    v->sN = t->stride[0];
    v->s1 = (int32_t)t->stride[1];
    v->s2 = (int32_t)t->stride[2];
    v->s3 = (int32_t)t->stride[3];
    return PWS_OK;
}

constexpr int64_t kAny = -1;   // check_arg: any size, dtype or device

// One tensor argument: present, a valid view, sizes (a, b, c, d), `dtype` and memory on device `dev`; kAny skips a check.
int check_arg(const pws_tensor *t, const char *what, int k, int64_t a, int64_t b, int64_t c, int64_t d, int dtype, int dev,
              View *v)
{
    PWS_TRY(make_view(t, what, k, v));
    const int64_t want[4] = {a, b, c, d};
    for (int i = 0; i < 4; ++i)
        if (want[i] != kAny && t->size[i] != want[i])
            return arg_error(PWS_EINVAL, what, k, "expected sizes [%lld, %lld, %lld, %lld], got [%lld, %lld, %lld, %lld] "
                             "(batch/channels or spatial sizes differ from the call's)", (long long)a, (long long)b,
                             (long long)c, (long long)d, (long long)t->size[0], (long long)t->size[1],
                             (long long)t->size[2], (long long)t->size[3]);
    if (dtype != kAny && t->dtype != dtype)
        return arg_error(PWS_EINVAL, what, k, "expected dtype %s, got %s", dtype_name(dtype), dtype_name(t->dtype));
    if (dev != kAny && t->device != dev) return arg_error(PWS_EINVAL, what, k, "expected device cuda:%d, got cuda:%d", dev, t->device);
    return PWS_OK;
}

// grad_input: the dense (N,C,H,W) buffer the library zero-fills and scatters into, on the frame's device; f32 (16-bit frames
// accumulate in fp32) or f64 for f64 frames.  An empty buffer (N*C = 0) is dense whatever its strides: torch keeps
// (H*W, H*W, W, 1) for C = 0.
int check_gin(const pws_tensor *gin, const pws_tensor *in, View *v)
{
    const int64_t Nb = in->size[0], C = in->size[1], H = in->size[2], W = in->size[3];
    PWS_TRY(check_arg(gin, "grad_input", -1, Nb, C, H, W, in->dtype == PWS_F64 ? PWS_F64 : PWS_F32, in->device, v));
    const bool dense = Nb * C == 0 || (gin->stride[3] == 1 && gin->stride[2] == W && gin->stride[1] == H * W &&
                                        (gin->stride[0] == C * H * W || Nb <= 1));
    if (!dense) return arg_error(PWS_EINVAL, "grad_input", -1, "must be (N,C,H,W)-contiguous (the library zero-fills it)");
    v->sN = C * H * W;
    return PWS_OK;
}

int check_modes(int interp, int padding)
{
    if (interp < 0 || interp > 2) { set_error("grid_sampler(): invalid interpolation mode %d", interp); return PWS_EINVAL; }
    if (padding < 0 || padding > 2) { set_error("grid_sampler(): invalid padding mode %d", padding); return PWS_EINVAL; }
    if (interp != PWS_INTERP_BILINEAR) {
        set_error("pwswarp: only mode='bilinear' is implemented (got interpolation_mode=%d)", interp);
        return PWS_EUNSUPPORTED;
    }
    if (padding == PWS_PAD_REFLECTION) {
        set_error("pwswarp: padding_mode='reflection' is not implemented (zeros and border only)");
        return PWS_EUNSUPPORTED;
    }
    return PWS_OK;
}

int check_spatial(const pws_tensor *in)
{
    for (int d = 2; d < 4; ++d)
        if (in->size[d] <= 0) {
            set_error("grid_sampler(): expected input to have non-empty spatial dimensions, but input has sizes [%lld, %lld, %lld, %lld] with dimension %d being empty",
                      (long long)in->size[0], (long long)in->size[1], (long long)in->size[2], (long long)in->size[3], d);
            return PWS_EINVAL;
        }
    return PWS_OK;
}

int check_pair(const pws_tensor *in, const pws_tensor *grid)
{
    if (!in || !grid) { set_error("grid_sampler(): expected input and grid to not be undefined"); return PWS_EINVAL; }
    if (in->device != grid->device) {
        set_error("grid_sampler(): expected input and grid to be on same device, but input is on cuda:%d and grid is on cuda:%d",
                  in->device, grid->device);
        return PWS_EINVAL;
    }
    if (in->size[0] != grid->size[0]) {
        set_error("grid_sampler(): expected grid and input to have same batch size, but got input with sizes [%lld, %lld, %lld, %lld] and grid with sizes [%lld, %lld, %lld, %lld]",
                  (long long)in->size[0], (long long)in->size[1], (long long)in->size[2], (long long)in->size[3],
                  (long long)grid->size[0], (long long)grid->size[1], (long long)grid->size[2], (long long)grid->size[3]);
        return PWS_EINVAL;
    }
    if (grid->size[3] != 2) {
        set_error("grid_sampler(): expected grid to have size 2 in last dimension, but got grid with sizes [%lld, %lld, %lld, %lld]",
                  (long long)grid->size[0], (long long)grid->size[1], (long long)grid->size[2], (long long)grid->size[3]);
        return PWS_EINVAL;
    }
    return check_spatial(in);
}

// frame: (N, C, H, W) sizes; (Ho, Wo): the output / map size
Geometry geometry(const int64_t (&frame)[4], int64_t Ho, int64_t Wo, int padding, int align)
{
    Geometry g;
    g.N = (int32_t)frame[0]; g.C = (int32_t)frame[1]; g.H = (int32_t)frame[2]; g.W = (int32_t)frame[3];
    g.Ho = (int32_t)Ho; g.Wo = (int32_t)Wo;
    g.padding = padding; g.align = align ? 1 : 0;
    return g;
}

// Whether a (pre_add, pre_mul, post_div, post_add) scale does anything before and after the sample; post_div must not be 0.
int scale_flags(float pre_add, float pre_mul, float post_div, float post_add, const char *what, int *has_pre, int *has_post)
{
    if (post_div == 0.0f) { set_error("%s: post_div must not be 0", what); return PWS_EINVAL; }
    *has_pre = !(pre_add == 0.0f && pre_mul == 1.0f);
    *has_post = !(post_div == 1.0f && post_add == 0.0f);
    return PWS_OK;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Runs launch() with `dev` selected (the caller's device is restored after) and reports its launch error as `what`'s.
template <class Launch>
int on_device(int dev, const char *what, Launch &&launch)
{
    DeviceGuard dg(dev);
    if (!dg.ok) { set_error("%s: cannot select cuda:%d", what, dev); return PWS_ECUDA; }
    PWS_TRY(launch());
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e)); return PWS_ECUDA; }
    return PWS_OK;
}

// Elements of a buffer that fills its span exactly, with no gap and no overlap, its dims in any stride order (so the
// planar-permuted maps torch hands over qualify); -1 for any other layout.
int64_t dense_numel(const pws_tensor *t)
{
    int64_t numel = 1, st[4], sz[4];
    int n = 0;
    for (int d = 0; d < 4; ++d) {
        numel *= t->size[d];
        if (t->size[d] == 1) continue;
        int i = n++;   // insertion by stride
        for (; i > 0 && st[i - 1] > t->stride[d]; --i) { st[i] = st[i - 1]; sz[i] = sz[i - 1]; }
        st[i] = t->stride[d]; sz[i] = t->size[d];
    }
    if (numel == 0) return 0;
    int64_t expected = 1;
    for (int i = 0; i < n; expected *= sz[i++])
        if (st[i] != expected) return -1;
    return numel;
}

// A backward with nothing to scatter (N*C*Ho*Wo == 0): every gradient the caller passed is defined and zero, as ATen
// returns it.  The buffers are dense (grad_input and glattice by their rules), so each takes one memset over its span.
int zero_grads(int dev, const char *what, cudaStream_t st, const pws_tensor *gin, const pws_tensor *const *ggrids, int K,
               bool staged, const pws_tensor *glattice, float *gtheta, int64_t N)
{
    if (N == 0) return PWS_OK;
    for (int k = 0; k < K; ++k)
        if (ggrids[k] && dense_numel(ggrids[k]) < 0)
            return arg_error(PWS_EUNSUPPORTED, "grad_grid", staged ? k : -1,
                             "with C = 0 the library zero-fills it, which needs a buffer without gaps");
    return on_device(dev, what, [&] {
        cudaError_t e = cudaSuccess;
        auto zero = [&](const pws_tensor *t) {
            if (t && e == cudaSuccess) e = cudaMemsetAsync(t->data, 0, (size_t)dense_numel(t) * elem_size(t->dtype), st);
        };
        zero(gin);
        for (int k = 0; k < K; ++k) zero(ggrids[k]);
        zero(glattice);
        if (gtheta && e == cudaSuccess) e = cudaMemsetAsync(gtheta, 0, (size_t)N * 6 * sizeof(float), st);
        if (e != cudaSuccess) { set_error("%s: cudaMemsetAsync: %s", what, cudaGetErrorString(e)); return (int)PWS_ECUDA; }
        return (int)PWS_OK;
    });
}

}  // namespace

static int make_scale(float pre_add, float pre_mul, float post_div, float post_add, StageScale *sc)
{
    PWS_TRY(scale_flags(pre_add, pre_mul, post_div, post_add, "stages", &sc->has_pre, &sc->has_post));
    sc->pre_add = pre_add; sc->pre_mul = pre_mul;
    sc->post_mul = 1.0f / post_div;   // fp32 division: the reciprocal torch's `tensor / scalar` kernel multiplies by
    sc->post_add = post_add;
    return PWS_OK;
}

// warp_stages dtype matrix: f32 frames with f32 maps; f16 / bf16 frames with f32 maps or maps of the frame's type; one map
// dtype for all stages.  Outputs and grad_outputs have the frame's dtype, grad_grids the maps'.
static int check_stage_dtypes(const pws_tensor *in, const pws_tensor *const *grids, int n_stages, const char *what)
{
    const bool half_in = in->dtype == PWS_F16 || in->dtype == PWS_BF16;
    if (in->dtype != PWS_F32 && !half_in) { set_error("%s: frames must be f32, f16 or bf16", what); return PWS_EUNSUPPORTED; }
    for (int k = 0; k < n_stages; ++k) {
        if (!grids[k]) { set_error("grid_sampler(): expected input and grid to not be undefined"); return PWS_EINVAL; }
        if (grids[k]->dtype != grids[0]->dtype) { set_error("%s: all maps must have one dtype (map 0: %d, map %d: %d)", what, grids[0]->dtype, k, grids[k]->dtype); return PWS_EINVAL; }
    }
    if (grids[0]->dtype != in->dtype && !(half_in && grids[0]->dtype == PWS_F32)) {
        set_error("%s: maps must be f32 or the frame's dtype (frame %d, maps %d)", what, in->dtype, grids[0]->dtype);
        return PWS_EINVAL;
    }
    return PWS_OK;
}

// The per-stage arguments of warp_stages: K maps of one size, and each stage's output (forward) or grad_output and optional
// grad_grid (backward; ggrids == nullptr for the forward).
static int check_stages(const pws_tensor *in, const pws_tensor *const *grids, const pws_tensor *const *io, const char *io_what,
                        const pws_tensor *const *ggrids, int K, const char *what, StageViews *sv)
{
    if (K < 1 || K > kMaxStages) { set_error("%s: n_stages must be 1..%d", what, kMaxStages); return PWS_EINVAL; }
    PWS_TRY(check_stage_dtypes(in, grids, K, what));
    const int64_t Nb = in->size[0], Ho = grids[0]->size[1], Wo = grids[0]->size[2];
    for (int k = 0; k < K; ++k) {
        PWS_TRY(check_pair(in, grids[k]));
        PWS_TRY(check_arg(grids[k], "grid", k, Nb, Ho, Wo, 2, kAny, in->device, &sv->map[k]));
        PWS_TRY(check_arg(io[k], io_what, k, Nb, in->size[1], Ho, Wo, in->dtype, in->device, &sv->io[k]));
        if (ggrids && ggrids[k]) PWS_TRY(check_arg(ggrids[k], "grad_grid", k, Nb, Ho, Wo, 2, grids[k]->dtype, in->device, &sv->gg[k]));
    }
    return PWS_OK;
}

int launch_forward_fused(const View &in, int in_dtype, const MapSpec &m, const View &out, int out_dtype,
                         const Geometry &g, cudaStream_t st);
int launch_compose_map(const MapSpec &m, const View &out, int N, int Ho, int Wo, cudaStream_t st);
int launch_backward_fused(const View &gout, const View &in, int in_dtype, const MapSpec &m, const View &gin, bool want_gin,
                          float *glat, float *gtheta, const Geometry &g, cudaStream_t st);

// dev: the call's device, where the drift must live
static int make_spec(const pws_map_spec *spec, int64_t N, int64_t Ho, int64_t Wo, int dev, MapSpec *m)
{
    if (!spec) { set_error("map spec: null"); return PWS_EINVAL; }
    if (spec->base < 0 || spec->base > 2 || spec->upsample < 0 || spec->upsample > 2) { set_error("map spec: bad base/upsample enum"); return PWS_EINVAL; }
    if (spec->map_h <= 0 || spec->map_w <= 0 || spec->map_h > INT_MAX || spec->map_w > INT_MAX) { set_error("map spec: bad lattice size"); return PWS_EINVAL; }
    m->drift.p = nullptr; m->drift.sN = 0; m->drift.s1 = m->drift.s2 = m->drift.s3 = 0;
    m->drift_dtype = PWS_F32;
    if (spec->drift) {
        const int dt = spec->drift->dtype;
        if (dt != PWS_F32 && dt != PWS_F16 && dt != PWS_BF16) { set_error("map spec: drift must be f32, f16 or bf16"); return PWS_EUNSUPPORTED; }
        m->drift_dtype = dt;
        PWS_TRY(check_arg(spec->drift, "drift", -1, N, spec->map_h, spec->map_w, 2, kAny, dev, &m->drift));
    } else if (spec->base == PWS_BASE_NONE) { set_error("map spec: no drift and no base"); return PWS_EINVAL; }
    if (spec->base == PWS_BASE_AFFINE && !spec->theta) { set_error("map spec: affine base needs theta"); return PWS_EINVAL; }
    if (spec->upsample == PWS_UP_NONE && (spec->map_h != Ho || spec->map_w != Wo)) {
        set_error("map spec: lattice %lldx%lld differs from the output %lldx%lld and no upsample was requested",
                  (long long)spec->map_h, (long long)spec->map_w, (long long)Ho, (long long)Wo);
        return PWS_EINVAL;
    }
    PWS_TRY(scale_flags(spec->pre_add, spec->pre_mul, spec->post_div, spec->post_add, "map spec", &m->has_pre, &m->has_post));
    m->theta = spec->theta; m->base = spec->base; m->base_align = spec->base_align_corners ? 1 : 0;
    m->upsample = spec->upsample; m->mh = (int)spec->map_h; m->mw = (int)spec->map_w;
    m->pre_add = spec->pre_add; m->pre_mul = spec->pre_mul; m->post_div = spec->post_div; m->post_add = spec->post_add;
    return PWS_OK;
}
}  // namespace pws

using namespace pws;

extern "C" {

__attribute__((visibility("default"))) int pws_abi_version(void) { return PWS_ABI_VERSION; }

__attribute__((visibility("default"))) const char *pws_last_error(void) { return g_err; }

__attribute__((visibility("default"))) uint64_t pws_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

__attribute__((visibility("default"))) const char *pws_last_kernel(void) { return g_last_kernel; }

__attribute__((visibility("default"))) int64_t pws_small_problem_elems(int64_t elems)
{
    if (elems < 0) return g_small_elems.load(std::memory_order_relaxed);
    return g_small_elems.exchange(elems, std::memory_order_relaxed);
}

__attribute__((visibility("default")))
int pws_warp2d_forward(const pws_tensor *in, const pws_tensor *grid, pws_tensor *out,
                       int interp, int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(interp, padding));
    PWS_TRY(check_pair(in, grid));
    Problem pb{};
    PWS_TRY(make_view(in, "input", -1, &pb.in));
    PWS_TRY(make_view(grid, "grid", -1, &pb.grid));
    const Geometry &g = pb.g = geometry(in->size, grid->size[1], grid->size[2], padding, align_corners);
    PWS_TRY(check_arg(out, "output", -1, g.N, g.C, g.Ho, g.Wo, in->dtype, in->device, &pb.out));
    pb.in_dtype = in->dtype; pb.grid_dtype = grid->dtype;
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return PWS_OK;
    return on_device(in->device, "forward", [&] { return launch_forward(pb, (cudaStream_t)stream); });
}

__attribute__((visibility("default")))
int pws_warp2d_backward(const pws_tensor *gout, const pws_tensor *in, const pws_tensor *grid,
                        pws_tensor *gin, pws_tensor *ggrid,
                        int interp, int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(interp, padding));
    PWS_TRY(check_pair(in, grid));
    Problem pb{};
    PWS_TRY(make_view(in, "input", -1, &pb.in));
    PWS_TRY(make_view(grid, "grid", -1, &pb.grid));
    const Geometry &g = pb.g = geometry(in->size, grid->size[1], grid->size[2], padding, align_corners);
    PWS_TRY(check_arg(gout, "grad_output", -1, g.N, g.C, g.Ho, g.Wo, in->dtype, in->device, &pb.gout));
    if (gin) PWS_TRY(check_gin(gin, in, &pb.gin));
    if (ggrid) PWS_TRY(check_arg(ggrid, "grad_grid", -1, g.N, g.Ho, g.Wo, 2, grid->dtype, in->device, &pb.ggrid));
    pb.want_gin = gin != nullptr;
    pb.want_ggrid = ggrid != nullptr;
    pb.in_dtype = in->dtype; pb.grid_dtype = grid->dtype;
    const cudaStream_t st = (cudaStream_t)stream;
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return zero_grads(in->device, "backward", st, gin, &ggrid, 1, false, nullptr, nullptr, g.N);
    return on_device(in->device, "backward", [&] { return launch_backward(pb, st); });
}

__attribute__((visibility("default")))
int pws_warp2d_taps(const pws_tensor *grid, int64_t in_h, int64_t in_w,
                    int32_t *x0, int32_t *y0, uint8_t *mask, float *weights,
                    int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!grid || !x0 || !y0 || !mask) { set_error("taps: null argument"); return PWS_EINVAL; }
    if (grid->dtype != PWS_F32) { set_error("taps: grid must be f32"); return PWS_EUNSUPPORTED; }
    if (grid->size[3] != 2) { set_error("taps: grid must have size 2 in its last dimension"); return PWS_EINVAL; }
    if (in_h <= 0 || in_w <= 0 || in_h > INT_MAX || in_w > INT_MAX) { set_error("taps: bad frame size"); return PWS_EINVAL; }
    View gv;
    PWS_TRY(make_view(grid, "grid", -1, &gv));
    const int64_t frame[4] = {grid->size[0], 1, in_h, in_w};
    const Geometry g = geometry(frame, grid->size[1], grid->size[2], padding, align_corners);
    return on_device(grid->device, "taps", [&] { return launch_taps(gv, g, x0, y0, mask, weights, (cudaStream_t)stream); });
}

__attribute__((visibility("default")))
int pws_warp2d_forward_fused(const pws_tensor *in, const pws_map_spec *spec, pws_tensor *out,
                             int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    View vin, vout;
    PWS_TRY(make_view(in, "input", -1, &vin));
    PWS_TRY(check_spatial(in));
    PWS_TRY(check_arg(out, "output", -1, in->size[0], in->size[1], kAny, kAny, kAny, in->device, &vout));
    const Geometry g = geometry(in->size, out->size[2], out->size[3], padding, align_corners);
    MapSpec m;
    PWS_TRY(make_spec(spec, g.N, g.Ho, g.Wo, in->device, &m));
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return PWS_OK;
    return on_device(in->device, "fused forward",
                     [&] { return launch_forward_fused(vin, in->dtype, m, vout, out->dtype, g, (cudaStream_t)stream); });
}

__attribute__((visibility("default")))
int pws_warp2d_backward_fused(const pws_tensor *gout, const pws_tensor *in, const pws_map_spec *spec,
                              pws_tensor *gin, pws_tensor *glattice, float *gtheta,
                              int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    View vin, vgout, vgin{}, vglat{};
    PWS_TRY(make_view(in, "input", -1, &vin));
    PWS_TRY(check_spatial(in));
    const bool half_in = in->dtype == PWS_F16 || in->dtype == PWS_BF16;
    if (in->dtype != PWS_F32 && in->dtype != PWS_U8 && !half_in) { set_error("fused backward: frames must be f32, f16, bf16 or uint8"); return PWS_EUNSUPPORTED; }
    if (gout && gout->dtype == PWS_U8) { set_error("fused backward: a uint8 output is not differentiable"); return PWS_EINVAL; }
    // grad_output has the forward output's dtype: f32 for f32 and uint8 frames, the frame's type for 16-bit frames
    PWS_TRY(check_arg(gout, "grad_output", -1, in->size[0], in->size[1], kAny, kAny, half_in ? in->dtype : PWS_F32, in->device,
                      &vgout));
    if (gtheta && (!spec || spec->base != PWS_BASE_AFFINE)) { set_error("fused backward: gtheta needs the affine base"); return PWS_EINVAL; }
    if (gtheta && !glattice) { set_error("fused backward: gtheta needs glattice (the library never allocates)"); return PWS_EINVAL; }
    const Geometry g = geometry(in->size, gout->size[2], gout->size[3], padding, align_corners);
    MapSpec m;
    PWS_TRY(make_spec(spec, g.N, g.Ho, g.Wo, in->device, &m));
    if (gin) {
        if (in->dtype == PWS_U8) { set_error("fused backward: a uint8 frame has no gradient (gin must be NULL)"); return PWS_EINVAL; }
        PWS_TRY(check_gin(gin, in, &vgin));
    }
    if (glattice) {
        PWS_TRY(check_arg(glattice, "glattice", -1, g.N, m.mh, m.mw, 2, PWS_F32, in->device, &vglat));
        const bool dense = glattice->stride[3] == 1 && glattice->stride[2] == 2 && glattice->stride[1] == 2 * m.mw &&
                           (glattice->stride[0] == 2 * m.mh * m.mw || g.N <= 1);
        if (!dense) { set_error("glattice: must be f32 (N,map_h,map_w,2)-contiguous (the library zero-fills it)"); return PWS_EINVAL; }
        // every node's (x, y) is stored, reduced into and read back as one 8-byte pair
        if (reinterpret_cast<uintptr_t>(glattice->data) & 7) { set_error("glattice: must be 8-byte aligned (one float2 per node)"); return PWS_EINVAL; }
    }
    const cudaStream_t st = (cudaStream_t)stream;
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return zero_grads(in->device, "fused backward", st, gin, nullptr, 0, false, glattice, gtheta, g.N);
    return on_device(in->device, "fused backward", [&] {
        return launch_backward_fused(vgout, vin, in->dtype, m, vgin, gin != nullptr, glattice ? (float *)glattice->data : nullptr,
                                     gtheta, g, st);
    });
}

__attribute__((visibility("default")))
int pws_compose_map(const pws_map_spec *spec, int64_t n, pws_tensor *map_out, void *stream)
{
    if (n < 0) { set_error("compose_map: negative n"); return PWS_EINVAL; }
    View vout;
    PWS_TRY(check_arg(map_out, "output", -1, n, kAny, kAny, 2, PWS_F32, kAny, &vout));
    MapSpec m;
    PWS_TRY(make_spec(spec, n, map_out->size[1], map_out->size[2], map_out->device, &m));
    return on_device(map_out->device, "compose_map", [&] {
        return launch_compose_map(m, vout, (int)n, (int)map_out->size[1], (int)map_out->size[2], (cudaStream_t)stream);
    });
}

__attribute__((visibility("default")))
int pws_warp2d_stages_forward(const pws_tensor *in, const pws_tensor *const *grids, pws_tensor *const *outs, int n_stages,
                              float pre_add, float pre_mul, float post_div, float post_add,
                              int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !grids || !outs) { set_error("stages forward: null argument"); return PWS_EINVAL; }
    View vin;
    PWS_TRY(make_view(in, "input", -1, &vin));
    StageViews sv{};
    PWS_TRY(check_stages(in, grids, outs, "output", nullptr, n_stages, "stages forward", &sv));
    const Geometry g = geometry(in->size, grids[0]->size[1], grids[0]->size[2], padding, align_corners);
    StageScale sc;
    PWS_TRY(make_scale(pre_add, pre_mul, post_div, post_add, &sc));
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return PWS_OK;
    return on_device(in->device, "stages forward", [&] {
        return launch_stages_forward(vin, in->dtype, sv, grids[0]->dtype, n_stages, g, sc, (cudaStream_t)stream);
    });
}

__attribute__((visibility("default")))
int pws_warp2d_stages_backward(const pws_tensor *const *gouts, const pws_tensor *in, const pws_tensor *const *grids,
                               pws_tensor *gin, pws_tensor *const *ggrids, int n_stages,
                               float pre_add, float pre_mul, float post_div, float post_add,
                               int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !grids || !gouts || !ggrids) { set_error("stages backward: null argument"); return PWS_EINVAL; }
    View vin, vgin{};
    PWS_TRY(make_view(in, "input", -1, &vin));
    StageViews sv{};
    PWS_TRY(check_stages(in, grids, gouts, "grad_output", ggrids, n_stages, "stages backward", &sv));
    if (gin) PWS_TRY(check_gin(gin, in, &vgin));
    const Geometry g = geometry(in->size, grids[0]->size[1], grids[0]->size[2], padding, align_corners);
    StageScale sc;
    PWS_TRY(make_scale(pre_add, pre_mul, post_div, post_add, &sc));
    const cudaStream_t st = (cudaStream_t)stream;
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0)
        return zero_grads(in->device, "stages backward", st, gin, ggrids, n_stages, true, nullptr, nullptr, g.N);
    return on_device(in->device, "stages backward", [&] {
        return launch_stages_backward(vin, in->dtype, sv, grids[0]->dtype, n_stages, vgin, gin != nullptr, g, sc, st);
    });
}

}  // extern "C"
