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

int make_view(const pws_tensor *t, const char *what, View *v)
{
    if (!t) { set_error("%s: null tensor descriptor", what); return PWS_EINVAL; }
    if (elem_size(t->dtype) == 0) { set_error("%s: unknown dtype %d", what, t->dtype); return PWS_EINVAL; }
    for (int d = 0; d < 4; ++d) {
        if (t->size[d] < 0) { set_error("%s: negative size", what); return PWS_EINVAL; }
        if (t->stride[d] < 0) { set_error("%s: negative strides are not supported", what); return PWS_EUNSUPPORTED; }
        if (t->size[d] > INT_MAX) { set_error("%s: dimension %d too large", what, d); return PWS_EUNSUPPORTED; }
    }
    if (item_span(t) >= ((int64_t)1 << 31)) {
        set_error("%s: one batch item spans >= 2^31 elements (32-bit in-frame offsets)", what);
        return PWS_EUNSUPPORTED;
    }
    const int64_t numel = t->size[0] * t->size[1] * t->size[2] * t->size[3];
    if (numel > 0 && !t->data) { set_error("%s: null data pointer", what); return PWS_EINVAL; }
    v->p = t->data;
    v->sN = t->stride[0];
    v->s1 = (int32_t)t->stride[1];
    v->s2 = (int32_t)t->stride[2];
    v->s3 = (int32_t)t->stride[3];
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
    for (int d = 2; d < 4; ++d)
        if (in->size[d] <= 0) {
            set_error("grid_sampler(): expected input to have non-empty spatial dimensions, but input has sizes [%lld, %lld, %lld, %lld] with dimension %d being empty",
                      (long long)in->size[0], (long long)in->size[1], (long long)in->size[2], (long long)in->size[3], d);
            return PWS_EINVAL;
        }
    return PWS_OK;
}

int fill_geometry(const pws_tensor *in, const pws_tensor *grid, int padding, int align, Geometry *g)
{
    g->N = (int32_t)in->size[0]; g->C = (int32_t)in->size[1];
    g->H = (int32_t)in->size[2]; g->W = (int32_t)in->size[3];
    g->Ho = (int32_t)grid->size[1]; g->Wo = (int32_t)grid->size[2];
    g->padding = padding; g->align = align ? 1 : 0;
    return PWS_OK;
}

int same_shape(const pws_tensor *t, int64_t a, int64_t b, int64_t c, int64_t d, const char *what)
{
    if (t->size[0] != a || t->size[1] != b || t->size[2] != c || t->size[3] != d) {
        set_error("%s: expected sizes [%lld, %lld, %lld, %lld], got [%lld, %lld, %lld, %lld]", what,
                  (long long)a, (long long)b, (long long)c, (long long)d,
                  (long long)t->size[0], (long long)t->size[1], (long long)t->size[2], (long long)t->size[3]);
        return PWS_EINVAL;
    }
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

int finish(const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e)); return PWS_ECUDA; }
    return PWS_OK;
}

}  // namespace
}  // namespace pws

namespace pws {
static int make_scale(float pre_add, float pre_mul, float post_div, float post_add, StageScale *sc)
{
    if (post_div == 0.0f) { set_error("stages: post_div must not be 0"); return PWS_EINVAL; }
    sc->pre_add = pre_add; sc->pre_mul = pre_mul;
    sc->post_mul = 1.0f / post_div;   // fp32 division: the reciprocal torch's `tensor / scalar` kernel multiplies by
    sc->post_add = post_add;
    sc->has_pre = !(pre_add == 0.0f && pre_mul == 1.0f);
    sc->has_post = !(post_div == 1.0f && post_add == 0.0f);
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

int launch_forward_fused(const View &in, int in_dtype, const MapSpec &m, const View &out, int out_dtype,
                         const Geometry &g, cudaStream_t st);
int launch_compose_map(const MapSpec &m, const View &out, int N, int Ho, int Wo, cudaStream_t st);
int launch_backward_fused(const View &gout, const View &in, int in_dtype, const MapSpec &m, const View &gin, bool want_gin,
                          float *glat, float *gtheta, const Geometry &g, cudaStream_t st);

static int make_spec(const pws_map_spec *spec, int64_t N, int64_t Ho, int64_t Wo, MapSpec *m)
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
        if (spec->drift->size[0] != N || spec->drift->size[1] != spec->map_h || spec->drift->size[2] != spec->map_w || spec->drift->size[3] != 2) {
            set_error("map spec: drift must have sizes [N, map_h, map_w, 2]"); return PWS_EINVAL;
        }
        int rc = make_view(spec->drift, "drift", &m->drift);
        if (rc != PWS_OK) return rc;
    } else if (spec->base == PWS_BASE_NONE) { set_error("map spec: no drift and no base"); return PWS_EINVAL; }
    if (spec->base == PWS_BASE_AFFINE && !spec->theta) { set_error("map spec: affine base needs theta"); return PWS_EINVAL; }
    if (spec->upsample == PWS_UP_NONE && (spec->map_h != Ho || spec->map_w != Wo)) {
        set_error("map spec: lattice %lldx%lld differs from the output %lldx%lld and no upsample was requested",
                  (long long)spec->map_h, (long long)spec->map_w, (long long)Ho, (long long)Wo);
        return PWS_EINVAL;
    }
    m->theta = spec->theta; m->base = spec->base; m->base_align = spec->base_align_corners ? 1 : 0;
    m->upsample = spec->upsample; m->mh = (int)spec->map_h; m->mw = (int)spec->map_w;
    m->pre_add = spec->pre_add; m->pre_mul = spec->pre_mul; m->post_div = spec->post_div; m->post_add = spec->post_add;
    m->has_pre = !(spec->pre_add == 0.0f && spec->pre_mul == 1.0f);
    m->has_post = !(spec->post_div == 1.0f && spec->post_add == 0.0f);
    if (spec->post_div == 0.0f) { set_error("map spec: post_div must not be 0"); return PWS_EINVAL; }
    return PWS_OK;
}
}  // namespace pws

using namespace pws;

#define PWS_TRY(expr) do { int rc_ = (expr); if (rc_ != PWS_OK) return rc_; } while (0)

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
    if (!out) { set_error("forward: null output descriptor"); return PWS_EINVAL; }
    Problem pb{};
    PWS_TRY(make_view(in, "input", &pb.in));
    PWS_TRY(make_view(grid, "grid", &pb.grid));
    PWS_TRY(make_view(out, "output", &pb.out));
    PWS_TRY(same_shape(out, in->size[0], in->size[1], grid->size[1], grid->size[2], "output"));
    if (out->dtype != in->dtype) { set_error("output: dtype must equal the input's"); return PWS_EINVAL; }
    if (out->device != in->device) { set_error("output: must be on the input's device"); return PWS_EINVAL; }
    fill_geometry(in, grid, padding, align_corners, &pb.g);
    pb.in_dtype = in->dtype; pb.grid_dtype = grid->dtype;
    if ((int64_t)pb.g.N * pb.g.C * pb.g.Ho * pb.g.Wo == 0) return PWS_OK;
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("forward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    PWS_TRY(launch_forward(pb, (cudaStream_t)stream));
    return finish("forward");
}

__attribute__((visibility("default")))
int pws_warp2d_backward(const pws_tensor *gout, const pws_tensor *in, const pws_tensor *grid,
                        pws_tensor *gin, pws_tensor *ggrid,
                        int interp, int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(interp, padding));
    PWS_TRY(check_pair(in, grid));
    if (!gout) { set_error("backward: null grad_output descriptor"); return PWS_EINVAL; }
    Problem pb{};
    PWS_TRY(make_view(in, "input", &pb.in));
    PWS_TRY(make_view(grid, "grid", &pb.grid));
    PWS_TRY(make_view(gout, "grad_output", &pb.gout));
    PWS_TRY(same_shape(gout, in->size[0], in->size[1], grid->size[1], grid->size[2], "grad_output"));
    if (gout->dtype != in->dtype) { set_error("grad_output: dtype must equal the input's"); return PWS_EINVAL; }
    if (gout->device != in->device) { set_error("grad_output: must be on the input's device"); return PWS_EINVAL; }
    pb.want_gin = gin != nullptr;
    pb.want_ggrid = ggrid != nullptr;
    if (gin) {
        PWS_TRY(make_view(gin, "grad_input", &pb.gin));
        PWS_TRY(same_shape(gin, in->size[0], in->size[1], in->size[2], in->size[3], "grad_input"));
        // 16-bit frames: grad_input is an fp32 accumulation buffer that the caller rounds once (see launch_16bit)
        const bool half_in = in->dtype == PWS_F16 || in->dtype == PWS_BF16;
        if ((half_in ? gin->dtype != PWS_F32 : gin->dtype != in->dtype) || gin->device != in->device) {
            set_error(half_in ? "grad_input: 16-bit frames accumulate into an f32 (N,C,H,W) buffer on the input's device"
                              : "grad_input: dtype/device must equal the input's");
            return PWS_EINVAL;
        }
        const int64_t C = in->size[1], H = in->size[2], W = in->size[3];
        const bool dense = gin->stride[3] == 1 && gin->stride[2] == W && gin->stride[1] == H * W &&
                           (gin->stride[0] == C * H * W || in->size[0] <= 1);
        if (!dense) { set_error("grad_input: must be (N,C,H,W)-contiguous (the library zero-fills it)"); return PWS_EINVAL; }
        pb.gin.sN = C * H * W;
    }
    if (ggrid) {
        PWS_TRY(make_view(ggrid, "grad_grid", &pb.ggrid));
        PWS_TRY(same_shape(ggrid, grid->size[0], grid->size[1], grid->size[2], 2, "grad_grid"));
        if (ggrid->dtype != grid->dtype || ggrid->device != in->device) { set_error("grad_grid: dtype/device must equal the grid's"); return PWS_EINVAL; }
    }
    fill_geometry(in, grid, padding, align_corners, &pb.g);
    pb.in_dtype = in->dtype; pb.grid_dtype = grid->dtype;
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("backward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    if (pb.g.N == 0) return PWS_OK;
    if ((int64_t)pb.g.C * pb.g.Ho * pb.g.Wo == 0) {
        // nothing scatters; grad_input is still defined (all zeros)
        if (gin && (int64_t)pb.g.C * pb.g.H * pb.g.W > 0) {
            cudaError_t e = cudaMemsetAsync(gin->data, 0, (size_t)(in->size[0] * pb.gin.sN * elem_size(gin->dtype)), (cudaStream_t)stream);
            if (e != cudaSuccess) { set_error("backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
        }
        return PWS_OK;
    }
    PWS_TRY(launch_backward(pb, (cudaStream_t)stream));
    return finish("backward");
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
    PWS_TRY(make_view(grid, "grid", &gv));
    Geometry g{};
    g.N = (int32_t)grid->size[0]; g.C = 1; g.H = (int32_t)in_h; g.W = (int32_t)in_w;
    g.Ho = (int32_t)grid->size[1]; g.Wo = (int32_t)grid->size[2];
    g.padding = padding; g.align = align_corners ? 1 : 0;
    DeviceGuard dg(grid->device);
    if (!dg.ok) { set_error("taps: cannot select cuda:%d", grid->device); return PWS_ECUDA; }
    PWS_TRY(launch_taps(gv, g, x0, y0, mask, weights, (cudaStream_t)stream));
    return finish("taps");
}

__attribute__((visibility("default")))
int pws_warp2d_forward_fused(const pws_tensor *in, const pws_map_spec *spec, pws_tensor *out,
                             int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !out) { set_error("fused forward: null tensor descriptor"); return PWS_EINVAL; }
    for (int d = 2; d < 4; ++d)
        if (in->size[d] <= 0) { set_error("grid_sampler(): expected input to have non-empty spatial dimensions"); return PWS_EINVAL; }
    if (out->size[0] != in->size[0] || out->size[1] != in->size[1]) { set_error("fused forward: output batch/channels must equal the input's"); return PWS_EINVAL; }
    if (out->device != in->device) { set_error("fused forward: output must be on the input's device"); return PWS_EINVAL; }
    View vin, vout;
    PWS_TRY(make_view(in, "input", &vin));
    PWS_TRY(make_view(out, "output", &vout));
    MapSpec m;
    PWS_TRY(make_spec(spec, in->size[0], out->size[2], out->size[3], &m));
    Geometry g{};
    g.N = (int32_t)in->size[0]; g.C = (int32_t)in->size[1]; g.H = (int32_t)in->size[2]; g.W = (int32_t)in->size[3];
    g.Ho = (int32_t)out->size[2]; g.Wo = (int32_t)out->size[3]; g.padding = padding; g.align = align_corners ? 1 : 0;
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return PWS_OK;
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("fused forward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    PWS_TRY(launch_forward_fused(vin, in->dtype, m, vout, out->dtype, g, (cudaStream_t)stream));
    return finish("fused forward");
}

__attribute__((visibility("default")))
int pws_warp2d_backward_fused(const pws_tensor *gout, const pws_tensor *in, const pws_map_spec *spec,
                              pws_tensor *gin, pws_tensor *glattice, float *gtheta,
                              int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !gout) { set_error("fused backward: null tensor descriptor"); return PWS_EINVAL; }
    for (int d = 2; d < 4; ++d)
        if (in->size[d] <= 0) { set_error("grid_sampler(): expected input to have non-empty spatial dimensions"); return PWS_EINVAL; }
    if (gout->size[0] != in->size[0] || gout->size[1] != in->size[1]) { set_error("fused backward: grad_output batch/channels must equal the input's"); return PWS_EINVAL; }
    if (gout->device != in->device) { set_error("fused backward: grad_output must be on the input's device"); return PWS_EINVAL; }
    const bool half_in = in->dtype == PWS_F16 || in->dtype == PWS_BF16;
    if (in->dtype != PWS_F32 && in->dtype != PWS_U8 && !half_in) { set_error("fused backward: frames must be f32, f16, bf16 or uint8"); return PWS_EUNSUPPORTED; }
    if (gout->dtype == PWS_U8) { set_error("fused backward: a uint8 output is not differentiable"); return PWS_EINVAL; }
    if (gout->dtype != (half_in ? in->dtype : PWS_F32)) {
        set_error("fused backward: grad_output must be f32 (f32 or uint8 frames) or the frame's 16-bit type (frame %d, grad_output %d)", in->dtype, gout->dtype);
        return PWS_EINVAL;
    }
    if (gtheta && (!spec || spec->base != PWS_BASE_AFFINE)) { set_error("fused backward: gtheta needs the affine base"); return PWS_EINVAL; }
    if (gtheta && !glattice) { set_error("fused backward: gtheta needs glattice (the library never allocates)"); return PWS_EINVAL; }
    View vin, vgout, vgin{}, vglat{};
    PWS_TRY(make_view(in, "input", &vin));
    PWS_TRY(make_view(gout, "grad_output", &vgout));
    MapSpec m;
    PWS_TRY(make_spec(spec, in->size[0], gout->size[2], gout->size[3], &m));
    if (gin) {
        if (in->dtype == PWS_U8) { set_error("fused backward: a uint8 frame has no gradient (gin must be NULL)"); return PWS_EINVAL; }
        PWS_TRY(make_view(gin, "grad_input", &vgin));
        PWS_TRY(same_shape(gin, in->size[0], in->size[1], in->size[2], in->size[3], "grad_input"));
        const int64_t C = in->size[1], H = in->size[2], W = in->size[3];
        const bool dense = gin->dtype == PWS_F32 && gin->stride[3] == 1 && gin->stride[2] == W && gin->stride[1] == H * W &&
                           (gin->stride[0] == C * H * W || in->size[0] <= 1);
        if (!dense) { set_error("grad_input: must be f32 (N,C,H,W)-contiguous (the library zero-fills it)"); return PWS_EINVAL; }
        if (gin->device != in->device) { set_error("fused backward: grad_input must be on the input's device"); return PWS_EINVAL; }
        vgin.sN = C * H * W;
    }
    if (glattice) {
        PWS_TRY(make_view(glattice, "glattice", &vglat));
        PWS_TRY(same_shape(glattice, in->size[0], spec->map_h, spec->map_w, 2, "glattice"));
        const int64_t h = spec->map_h, w = spec->map_w;
        const bool dense = glattice->dtype == PWS_F32 && glattice->stride[3] == 1 && glattice->stride[2] == 2 &&
                           glattice->stride[1] == 2 * w && (glattice->stride[0] == 2 * h * w || in->size[0] <= 1);
        if (!dense) { set_error("glattice: must be f32 (N,map_h,map_w,2)-contiguous (the library zero-fills it)"); return PWS_EINVAL; }
        // every node's (x, y) is stored, reduced into and read back as one 8-byte pair
        if (reinterpret_cast<uintptr_t>(glattice->data) & 7) { set_error("glattice: must be 8-byte aligned (one float2 per node)"); return PWS_EINVAL; }
        if (glattice->device != in->device) { set_error("fused backward: glattice must be on the input's device"); return PWS_EINVAL; }
    }
    Geometry g{};
    g.N = (int32_t)in->size[0]; g.C = (int32_t)in->size[1]; g.H = (int32_t)in->size[2]; g.W = (int32_t)in->size[3];
    g.Ho = (int32_t)gout->size[2]; g.Wo = (int32_t)gout->size[3]; g.padding = padding; g.align = align_corners ? 1 : 0;
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("fused backward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    if (g.N == 0) return PWS_OK;
    if ((int64_t)g.C * g.Ho * g.Wo == 0) {
        // nothing flows back; the gradients are still defined (all zeros)
        cudaStream_t st = (cudaStream_t)stream;
        cudaError_t e = cudaSuccess;
        if (gin && (int64_t)g.C * g.H * g.W > 0) e = cudaMemsetAsync(gin->data, 0, (size_t)(g.N * vgin.sN * 4), st);
        if (e == cudaSuccess && glattice) e = cudaMemsetAsync(glattice->data, 0, (size_t)g.N * m.mh * m.mw * 2 * 4, st);
        if (e == cudaSuccess && gtheta) e = cudaMemsetAsync(gtheta, 0, (size_t)g.N * 6 * 4, st);
        if (e != cudaSuccess) { set_error("fused backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
        return PWS_OK;
    }
    PWS_TRY(launch_backward_fused(vgout, vin, in->dtype, m, vgin, gin != nullptr, glattice ? (float *)glattice->data : nullptr,
                                  gtheta, g, (cudaStream_t)stream));
    return finish("fused backward");
}

__attribute__((visibility("default")))
int pws_compose_map(const pws_map_spec *spec, int64_t n, pws_tensor *map_out, void *stream)
{
    if (!map_out) { set_error("compose_map: null output"); return PWS_EINVAL; }
    if (map_out->dtype != PWS_F32 || map_out->size[3] != 2 || map_out->size[0] != n) { set_error("compose_map: output must be f32 (N,Ho,Wo,2)"); return PWS_EINVAL; }
    View vout;
    PWS_TRY(make_view(map_out, "map_out", &vout));
    MapSpec m;
    PWS_TRY(make_spec(spec, n, map_out->size[1], map_out->size[2], &m));
    DeviceGuard dg(map_out->device);
    if (!dg.ok) { set_error("compose_map: cannot select cuda:%d", map_out->device); return PWS_ECUDA; }
    PWS_TRY(launch_compose_map(m, vout, (int)n, (int)map_out->size[1], (int)map_out->size[2], (cudaStream_t)stream));
    return finish("compose_map");
}

__attribute__((visibility("default")))
int pws_warp2d_stages_forward(const pws_tensor *in, const pws_tensor *const *grids, pws_tensor *const *outs, int n_stages,
                              float pre_add, float pre_mul, float post_div, float post_add,
                              int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !grids || !outs) { set_error("stages forward: null argument"); return PWS_EINVAL; }
    if (n_stages < 1 || n_stages > kMaxStages) { set_error("stages forward: n_stages must be 1..%d", kMaxStages); return PWS_EINVAL; }
    PWS_TRY(check_stage_dtypes(in, grids, n_stages, "stages forward"));
    View vin;
    PWS_TRY(make_view(in, "input", &vin));
    StageViews sv{};
    Geometry g{};
    for (int k = 0; k < n_stages; ++k) {
        PWS_TRY(check_pair(in, grids[k]));
        if (!outs[k]) { set_error("stages forward: null output %d", k); return PWS_EINVAL; }
        if (outs[k]->dtype != in->dtype) { set_error("stages forward: output %d: dtype must equal the input's", k); return PWS_EINVAL; }
        if (k && (grids[k]->size[1] != grids[0]->size[1] || grids[k]->size[2] != grids[0]->size[2])) { set_error("stages forward: all maps must have the same size"); return PWS_EINVAL; }
        PWS_TRY(make_view(grids[k], "grid", &sv.map[k]));
        PWS_TRY(make_view(outs[k], "output", &sv.io[k]));
        PWS_TRY(same_shape(outs[k], in->size[0], in->size[1], grids[k]->size[1], grids[k]->size[2], "output"));
        if (outs[k]->device != in->device) { set_error("stages forward: output must be on the input's device"); return PWS_EINVAL; }
    }
    fill_geometry(in, grids[0], padding, align_corners, &g);
    StageScale sc;
    PWS_TRY(make_scale(pre_add, pre_mul, post_div, post_add, &sc));
    if ((int64_t)g.N * g.C * g.Ho * g.Wo == 0) return PWS_OK;
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("stages forward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    PWS_TRY(launch_stages_forward(vin, in->dtype, sv, grids[0]->dtype, n_stages, g, sc, (cudaStream_t)stream));
    return finish("stages forward");
}

__attribute__((visibility("default")))
int pws_warp2d_stages_backward(const pws_tensor *const *gouts, const pws_tensor *in, const pws_tensor *const *grids,
                               pws_tensor *gin, pws_tensor *const *ggrids, int n_stages,
                               float pre_add, float pre_mul, float post_div, float post_add,
                               int padding, int align_corners, void *stream)
{
    PWS_TRY(check_modes(PWS_INTERP_BILINEAR, padding));
    if (!in || !grids || !gouts || !ggrids) { set_error("stages backward: null argument"); return PWS_EINVAL; }
    if (n_stages < 1 || n_stages > kMaxStages) { set_error("stages backward: n_stages must be 1..%d", kMaxStages); return PWS_EINVAL; }
    PWS_TRY(check_stage_dtypes(in, grids, n_stages, "stages backward"));
    View vin, vgin{};
    PWS_TRY(make_view(in, "input", &vin));
    StageViews sv{};
    Geometry g{};
    for (int k = 0; k < n_stages; ++k) {
        PWS_TRY(check_pair(in, grids[k]));
        if (!gouts[k]) { set_error("stages backward: null grad_output %d", k); return PWS_EINVAL; }
        if (gouts[k]->dtype != in->dtype) { set_error("stages backward: grad_output %d: dtype must equal the input's", k); return PWS_EINVAL; }
        if (gouts[k]->device != in->device) { set_error("stages backward: grad_output %d: must be on the input's device", k); return PWS_EINVAL; }
        if (k && (grids[k]->size[1] != grids[0]->size[1] || grids[k]->size[2] != grids[0]->size[2])) { set_error("stages backward: all maps must have the same size"); return PWS_EINVAL; }
        PWS_TRY(make_view(grids[k], "grid", &sv.map[k]));
        PWS_TRY(make_view(gouts[k], "grad_output", &sv.io[k]));
        PWS_TRY(same_shape(gouts[k], in->size[0], in->size[1], grids[k]->size[1], grids[k]->size[2], "grad_output"));
        if (ggrids[k]) {
            if (ggrids[k]->dtype != grids[k]->dtype) { set_error("stages backward: grad_grid %d: dtype must equal the map's", k); return PWS_EINVAL; }
            if (ggrids[k]->device != in->device) { set_error("stages backward: grad_grid %d: must be on the input's device", k); return PWS_EINVAL; }
            PWS_TRY(make_view(ggrids[k], "grad_grid", &sv.gg[k]));
            PWS_TRY(same_shape(ggrids[k], grids[k]->size[0], grids[k]->size[1], grids[k]->size[2], 2, "grad_grid"));
        }
    }
    if (gin) {
        PWS_TRY(make_view(gin, "grad_input", &vgin));
        PWS_TRY(same_shape(gin, in->size[0], in->size[1], in->size[2], in->size[3], "grad_input"));
        const int64_t C = in->size[1], H = in->size[2], W = in->size[3];
        const bool dense = gin->dtype == PWS_F32 && gin->stride[3] == 1 && gin->stride[2] == W && gin->stride[1] == H * W &&
                           (gin->stride[0] == C * H * W || in->size[0] <= 1);
        if (!dense) {
            set_error("grad_input: must be f32 (N,C,H,W)-contiguous (the library zero-fills it; 16-bit frames accumulate in fp32)");
            return PWS_EINVAL;
        }
        if (gin->device != in->device) { set_error("stages backward: grad_input must be on the input's device"); return PWS_EINVAL; }
        vgin.sN = C * H * W;
    }
    fill_geometry(in, grids[0], padding, align_corners, &g);
    StageScale sc;
    PWS_TRY(make_scale(pre_add, pre_mul, post_div, post_add, &sc));
    DeviceGuard dg(in->device);
    if (!dg.ok) { set_error("stages backward: cannot select cuda:%d", in->device); return PWS_ECUDA; }
    if (g.N == 0) return PWS_OK;
    if ((int64_t)g.C * g.Ho * g.Wo == 0) {
        if (gin && (int64_t)g.C * g.H * g.W > 0) {
            cudaError_t e = cudaMemsetAsync(gin->data, 0, (size_t)(in->size[0] * vgin.sN * 4), (cudaStream_t)stream);
            if (e != cudaSuccess) { set_error("stages backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return PWS_ECUDA; }
        }
        return PWS_OK;
    }
    PWS_TRY(launch_stages_backward(vin, in->dtype, sv, grids[0]->dtype, n_stages, vgin, gin != nullptr, g, sc, (cudaStream_t)stream));
    return finish("stages backward");
}

}  // extern "C"
