/*
 * pwswarp.h -- C ABI of libpwswarp.so, the B200 (sm_100a) pixel-wise bilinear warp.
 *
 * This is the drop-in boundary for ONE path of mindazhao/PWStableNet: the
 * torch.nn.functional.grid_sample calls that resample each unstable frame by the
 * per-pixel map netG produced (R = the reference checkout):
 *     R/main_new.py:106,109,116,118   training warps, RGB x3 stages x2 clips + gray
 *     R/main_new.py:197               chained affine warp (gradient flows to the frame)
 *     R/main_new.py:716               inference warp at native video resolution
 *     R/main.py:106,107,114,115,319,325,643   the stale twins
 *     R/main_new.py:214               loss_g.backward() -> grid_sampler_2d_backward
 * What sits underneath those calls in the reference is ATen:
 *     aten::grid_sampler_2d(Tensor input, Tensor grid, int interpolation_mode,
 *                           int padding_mode, bool align_corners) -> Tensor
 *     aten::grid_sampler_2d_backward(Tensor grad_output, Tensor input, Tensor grid, int, int, bool,
 *                           bool[2] output_mask) -> (Tensor, Tensor)
 * ($TORCH/include/ATen/native/cuda/GridSampler.h:12-24 is the launcher pair the
 * two entry points below replace.)  Enumerations are numerically identical to
 * ATen's (GridSamplerUtils.h:14-15).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types, no C++ exceptions across the ABI
 *   - every buffer is caller-owned DEVICE memory; the library never allocates,
 *     frees or retains a pointer past the call
 *   - strides are in ELEMENTS and arbitrary (permuted / sliced views are the norm:
 *     the reference passes planar-stored maps, strides (2HW, W, 1, HW))
 *   - asynchronous on `stream` (a cudaStream_t; NULL = legacy default stream)
 *   - return 0 on success, negative pws_status on failure; the message is in the
 *     thread-local pws_last_error()
 *   - every tensor argument, the map spec's drift included, must live on the frame's
 *     device (pws_compose_map: on map_out's device); theta / gtheta are raw pointers
 *     the library cannot check
 *   - stateless and re-entrant
 */
#ifndef PWSWARP_H_
#define PWSWARP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PWS_ABI_VERSION 1

typedef enum pws_dtype {
    PWS_F32 = 0,
    PWS_F16 = 1,
    PWS_BF16 = 2,
    PWS_F64 = 3,
    PWS_U8 = 4,
    PWS_I32 = 5
} pws_dtype;

typedef enum pws_status {
    PWS_OK = 0,
    PWS_EINVAL = -1,       /* bad shape / stride / pointer / enum: ValueError-class */
    PWS_EUNSUPPORTED = -2, /* valid for torch, outside this library's scope (SURVEY 8(b)) */
    PWS_ECUDA = -3         /* a CUDA runtime call failed */
} pws_status;

/* ATen GridSamplerInterpolation / GridSamplerPadding */
enum { PWS_INTERP_BILINEAR = 0, PWS_INTERP_NEAREST = 1, PWS_INTERP_BICUBIC = 2 };
enum { PWS_PAD_ZEROS = 0, PWS_PAD_BORDER = 1, PWS_PAD_REFLECTION = 2 };

/* A 4-D strided view of device memory.
 *   frames / outputs / grad_output / grad_input : (N, C, H, W)
 *   maps  / grad_grid                            : (N, H_out, W_out, 2)   [..., 0] = x, [..., 1] = y */
typedef struct pws_tensor {
    void *data;
    int32_t dtype;  /* pws_dtype */
    int32_t device; /* CUDA ordinal the memory lives on */
    int64_t size[4];
    int64_t stride[4];
} pws_tensor;

int pws_abi_version(void);

/* Thread-local, valid until the next failing call on the same thread. */
const char *pws_last_error(void);

/* Number of CUDA kernels this library has launched in this process (all threads).
 * bench.py reports the difference over its timed region as "gpu_launches". */
uint64_t pws_launch_count(void);

/* Debug / tests: name of the kernel family the last forward / backward call on THIS thread launched
 * ("fwd_tma", "fwd_lean", "fwd_direct", "bwd_tma", "bwd_lean", "bwd_march", "bwd_lean_16", "bwd_march_16", "fwd_fused",
 * "stages_fwd", "stages_fwd_16", ...; "" before any call). */
const char *pws_last_kernel(void);

/* Tuning knob (process-wide, like a library's "benchmark" switch; results do not depend on it): calls whose output has at
 * most this many elements -- the whole working set sits in L2, the call is bound by its launch -- take the plain one-wave
 * kernels instead of the persistent TMA pipelines.  Returns the previous value; a negative argument only queries.
 * Default 4 Mi elements (the reference's 16 x 3 x 256 x 256 training shapes are 3 Mi).  0 = always the TMA pipelines
 * (the test-suite uses that to reach them with small inputs). */
int64_t pws_small_problem_elems(int64_t elems);

/* out[n,c,h,w] = sum over the 4 bilinear taps of in[n,c,y_tap,x_tap] * w_tap,
 * replaces aten::grid_sampler_2d for interp = bilinear, padding in {zeros, border}.
 * Frame dtype: f32, f16, bf16, f64.  Map dtype: the frame's dtype or f32 (an
 * extension torch does not offer: 16-bit frames with fp32 maps, BASELINE config 5).
 * `out` has the frame dtype; arithmetic is fp32 (fp64 for f64), in ATen's CUDA
 * operation order, so fp32 results are bit-identical to torch's CUDA kernel. */
int pws_warp2d_forward(const pws_tensor *in, const pws_tensor *grid, pws_tensor *out,
                       int interp, int padding, int align_corners, void *stream);

/* Replaces aten::grid_sampler_2d_backward.  gin / ggrid may be NULL
 * (== output_mask[0] / [1] false).  gin must be a dense (N,C,H,W)-contiguous
 * buffer; it does NOT need to arrive zeroed: the library zero-fills it itself,
 * frame by frame, just ahead of the scatter so the lines are still in L2 when
 * the atomics land (DESIGN.md "backward").  ggrid is fully overwritten.
 * With C = 0 nothing flows back: gin and ggrid are zero-filled, as ATen returns them.
 * That takes one memset over each buffer, so ggrid must then be dense in some order of
 * its dims (interleaved, or the planar-permuted layout); any other layout is
 * PWS_EUNSUPPORTED.  gin may keep any strides when it is empty (N*C = 0).
 * Accepts every (frame, map) dtype pair pws_warp2d_forward accepts, any strides and C:
 *     frame / gout   map / ggrid     gin
 *     f32            f32             f32
 *     f64            f64             f64
 *     f16 | bf16     f32             f32
 *     f16 | bf16     the frame's     f32
 * For 16-bit frames the arithmetic is fp32: ggrid is the fp32 result rounded once to
 * the map's dtype, and gin is an fp32 ACCUMULATION buffer holding the exact fp32
 * sums, which the caller rounds to the frame dtype once (16-bit atomics would round
 * after every add). */
int pws_warp2d_backward(const pws_tensor *gout, const pws_tensor *in, const pws_tensor *grid,
                        pws_tensor *gin, pws_tensor *ggrid,
                        int interp, int padding, int align_corners, void *stream);

/* Debug / parity entry: the north-west tap (x0, y0), the 4-bit validity mask
 * (bit0 nw, bit1 ne, bit2 sw, bit3 se) and optionally the four weights the forward
 * pass uses for every output pixel.  x0, y0: int32 (N,Ho,Wo) contiguous; mask: uint8
 * (N,Ho,Wo) contiguous; weights: float (N,Ho,Wo,4) contiguous or NULL.
 * grid must be f32. */
int pws_warp2d_taps(const pws_tensor *grid, int64_t in_h, int64_t in_w,
                    int32_t *x0, int32_t *y0, uint8_t *mask, float *weights,
                    int padding, int align_corners, void *stream);

/* ---- map composition fused into the sample (SURVEY.md 8(a) rows a7-a11) -------------------
 * The map is not read from memory but composed per output pixel:
 *     lattice(i,j) = drift[n,i,j,:] + base(i,j)            on a (map_h x map_w) lattice
 *     map(h,w)     = lattice(h,w)                           upsample == PWS_UP_NONE
 *                  = bilinear resize of the lattice         PWS_UP_ALIGNED   (nn.UpsamplingBilinear2d,
 *                    to the output size                                       R/main_new.py:706-710)
 *                                                           PWS_UP_HALF_PIXEL (nn.Upsample(mode='bilinear'),
 *                                                                             R/main.py:639-641)
 * base: PWS_BASE_NONE      drift already is the map
 *       PWS_BASE_IDENTITY  generate_maps' meshgrid X*2/(W-1)-1          (R/lib/utils.py:386-403)
 *       PWS_BASE_AFFINE    F.affine_grid(theta, size, base_align_corners) (R/lib/networks_cascading.py:164,235)
 * Around the sample: frame' = (frame + pre_add) * pre_mul, out = acc / post_div + post_add
 * (R/main_new.py:106-107: (x+1)*127.5 ... /127.5-1); (0,1,1,0) switches them off.
 * Frames may be PWS_U8 (cv2 HWC buffers, R/main_new.py:679-684) and the output PWS_U8
 * (truncating store, R/main_new.py:717-721), PWS_F32, or the frame's 16-bit float type. */
enum { PWS_BASE_NONE = 0, PWS_BASE_IDENTITY = 1, PWS_BASE_AFFINE = 2 };
enum { PWS_UP_NONE = 0, PWS_UP_ALIGNED = 1, PWS_UP_HALF_PIXEL = 2 };

typedef struct pws_map_spec {
    const pws_tensor *drift; /* (N, map_h, map_w, 2) f32, f16 or bf16 view, any strides; NULL = zero drift.  A 16-bit
                                drift is upcast exactly: results equal those of the same call with its f32 copy */
    const float *theta;      /* (N,2,3) f32 contiguous device memory; PWS_BASE_AFFINE only */
    int32_t base;
    int32_t base_align_corners;
    int32_t upsample;
    int32_t reserved;
    int64_t map_h, map_w;
    float pre_add, pre_mul, post_div, post_add;
} pws_map_spec;

/* Forward warp with the composed map; `out` (N,C,Ho,Wo) fixes the output size.
 * Arithmetic is fp32 for every frame type (uint8 and 16-bit frames are upcast exactly): (x + pre_add) * pre_mul per tap,
 * the bilinear sample in ATen's order, acc / post_div (a true division) + post_add, each op rounded in fp32.  The result
 * is rounded ONCE, at the store: to the output's 16-bit type (round to nearest even), or for a PWS_U8 output clamped to
 * [0, 255] and truncated (NaN -> 0).  This differs on purpose from pws_warp2d_stages_forward, which reproduces torch's
 * rounding to the frame type after every elementwise op: warp_fused replaces an inference pipeline whose intermediates
 * were fp32, and one rounding is the closer result. */
int pws_warp2d_forward_fused(const pws_tensor *in, const pws_map_spec *spec, pws_tensor *out,
                             int padding, int align_corners, void *stream);

/* Autograd of pws_warp2d_forward_fused.  spec, padding and align_corners are what the forward was given; gout has the
 * forward output's sizes (any strides) and dtype, which must be a float one: f32 for f32 and uint8 frames, the frame's
 * type for f16 / bf16 frames (a uint8 output is not differentiable: PWS_EINVAL).  Every output is optional (NULL):
 *     gin       (N,C,H,W) dense f32 accumulation buffer, zero-filled by the library; the caller rounds it to the frame
 *               dtype once.  Not for uint8 frames.
 *     glattice  (N,map_h,map_w,2) dense f32, 8-byte aligned (each node's pair is one 8-byte access), zero-filled by
 *               the library: d loss / d lattice, which is d loss / d drift (the drift enters additively); also allowed
 *               without a drift.
 *     gtheta    (N,2,3) f32 contiguous device memory, PWS_BASE_AFFINE only, needs glattice:
 *               gtheta[n,c,:] = sum_ij glattice[n,i,j,c] * (bx_j, by_i, 1), with the base coordinates the forward uses.
 * The map is recomputed with the forward's statements (same taps); go = gout / post_div (a true division, as the forward
 * divides); grad_grid follows ATen's statement order on the pre-scaled taps; fp32 throughout.  Without upsample glattice
 * equals pws_warp2d_backward's grad_grid of the composed map bit for bit; with upsample it is that grad_grid pushed
 * through the upsample's adjoint, summed with atomics (order-dependent in the last bits).  With C = 0 every output given
 * is zero-filled. */
int pws_warp2d_backward_fused(const pws_tensor *gout, const pws_tensor *in, const pws_map_spec *spec,
                              pws_tensor *gin, pws_tensor *glattice, float *gtheta,
                              int padding, int align_corners, void *stream);

/* Debug / parity: writes the map the fused kernel uses into map_out (N,Ho,Wo,2) f32 (also for a 16-bit drift). */
int pws_compose_map(const pws_map_spec *spec, int64_t n, pws_tensor *map_out, void *stream);

/* ---- K maps, one frame, one launch (SURVEY.md 8(a) rows a8, a11; north_star "map composition across cascade
 * stages fused into the sample") ---------------------------------------------------------------------------------
 * Replaces the reference's per-stage sequence R/main_new.py:103-110 (and :112-119)
 *     for nl in range(num_layer): fake[nl] = grid_sample((frame + 1) * 127.5, grid[nl]) / 127.5 - 1
 * and its autograd (R/main_new.py:214): every stage's map samples the SAME frame, which is read once; the scaled frame
 * and the unscaled samples never reach HBM.
 *     outs[k]   = sample((in + pre_add) * pre_mul, grids[k]) * (1 / post_div) + post_add        k < n_stages <= 4
 *     ggrids[k] = d outs[k] / d grids[k] applied to gouts[k]      (entries may be NULL)
 *     gin       = sum_k d outs[k] / d in applied to gouts[k]      (may be NULL; dense NCHW, zero-filled by the library)
 * With C = 0, gin and every ggrids[k] are zero-filled, under pws_warp2d_backward's layout rule for ggrid.
 * C in {1, 3}, any strides.  `1 / post_div` is the rounded fp32 reciprocal torch's `tensor / scalar` multiplies by, so
 * the results equal the reference's sequence of torch calls bit for bit.  (0, 1, 1, 0) switches the scales off.
 * dtypes (all grids share one dtype; anything else is PWS_EINVAL):
 *     in / outs / gouts   grids / ggrids     gin
 *     f32                 f32                f32
 *     f16 | bf16          f32                f32 accumulation buffer
 *     f16 | bf16          the frame's        f32 accumulation buffer
 * For 16-bit frames the results equal that sequence evaluated by torch on tensors of the frame's type, where every
 * elementwise op computes in fp32 and rounds to the type (round_T):
 *     tap  = round_T(round_T(x + pre_add) * pre_mul)                 (pre scale on)
 *     s    = round_T(fp32 bilinear sample of the taps, ATen's order)
 *     out  = round_T(round_T(s * (1 / post_div)) + post_add)          (post scale on)
 * The backward is that sequence's autograd through pws_warp2d_backward: go = round_T(gout * (1 / post_div)), fp32
 * arithmetic on the rounded taps, ggrid rounded once to the map's type; gin holds the exact fp32 sums (times pre_mul,
 * over all stages), which the caller rounds to the frame type once. */
int pws_warp2d_stages_forward(const pws_tensor *in, const pws_tensor *const *grids, pws_tensor *const *outs, int n_stages,
                              float pre_add, float pre_mul, float post_div, float post_add,
                              int padding, int align_corners, void *stream);
int pws_warp2d_stages_backward(const pws_tensor *const *gouts, const pws_tensor *in, const pws_tensor *const *grids,
                               pws_tensor *gin, pws_tensor *const *ggrids, int n_stages,
                               float pre_add, float pre_mul, float post_div, float post_add,
                               int padding, int align_corners, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PWSWARP_H_ */
