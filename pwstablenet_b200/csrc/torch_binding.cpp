// torch_binding.cpp -- the PyTorch caller's side of the C ABI in C++ (host code only; no kernels here).
//
// pwstablenet_b200.grid_sample is a torch.autograd.Function in Python (functional.py) that fills pws_tensor descriptors
// with ctypes.  At the reference's TRAINING shapes (R/main_new.py:106-118,197: 256 x 256 frames, per-GPU batch 16 down to 2
// under DDP) a warp is a 15-30 us kernel and the Python around it -- descriptor packing, torch.empty, the stream lookup,
// the Function machinery, twice per call site -- costs 120 us per forward + backward against 73 us for torch's own
// operator (tools/host_overhead.py on the B200 host).  This file is the same shim compiled: descriptors from
// at::Tensor, outputs from at::empty, the current stream from c10, the autograd node from torch::autograd::Function.  It calls
// the SAME exported entry points of libpwswarp.so (include/pwswarp.h) with the same arguments; nothing is computed here.
//
// Mirrors: aten::grid_sampler_2d / aten::grid_sampler_2d_backward ($TORCH/include/ATen/native/cuda/GridSampler.h:12-24),
// output allocation as ATen does it (forward: NCHW-contiguous; grad_input: like input, contiguous; grad_grid: like grid).
#include <torch/extension.h>
#include <c10/cuda/CUDAStream.h>

#include "../../include/pwswarp.h"

namespace {

int dtype_code(const at::Tensor &t)
{
    switch (t.scalar_type()) {
    case at::kFloat: return PWS_F32;
    case at::kHalf: return PWS_F16;
    case at::kBFloat16: return PWS_BF16;
    case at::kDouble: return PWS_F64;
    default: TORCH_CHECK_NOT_IMPLEMENTED(false, "pwstablenet_b200.grid_sample: unsupported dtype ", t.scalar_type());
    }
    return -1;
}

pws_tensor desc(const at::Tensor &t)
{
    pws_tensor d;
    d.data = t.data_ptr();
    d.dtype = dtype_code(t);
    d.device = (int32_t)t.get_device();
    for (int i = 0; i < 4; ++i) { d.size[i] = t.size(i); d.stride[i] = t.stride(i); }
    return d;
}

// pws_status -> the exception the Python shim raises (_lib.check)
void check(int rc)
{
    if (rc == PWS_OK) return;
    const char *msg = pws_last_error();
    if (rc == PWS_EUNSUPPORTED) TORCH_CHECK_NOT_IMPLEMENTED(false, msg);
    if (rc == PWS_EINVAL) TORCH_CHECK(false, msg);
    TORCH_CHECK(false, "pwswarp CUDA error: ", msg);
}

void *current_stream(const at::Tensor &t) { return c10::cuda::getCurrentCUDAStream(t.get_device()).stream(); }

at::Tensor warp2d_forward(const at::Tensor &input, const at::Tensor &grid, int64_t padding, bool align_corners)
{
    at::Tensor out = at::empty({input.size(0), input.size(1), grid.size(1), grid.size(2)}, input.options());
    const pws_tensor din = desc(input), dg = desc(grid);
    pws_tensor dout = desc(out);
    check(pws_warp2d_forward(&din, &dg, &dout, PWS_INTERP_BILINEAR, (int)padding, align_corners ? 1 : 0, current_stream(input)));
    return out;
}

// uninitialised tensor with t's sizes; keeps t's strides when they are dense (the reference's maps are planar-stored
// permuted views), otherwise contiguous -- functional._like_layout
at::Tensor like_layout(const at::Tensor &t)
{
    if (t.numel() > 0 && t.is_non_overlapping_and_dense()) return at::empty_strided(t.sizes(), t.strides(), t.options());
    return at::empty(t.sizes(), t.options());
}

std::tuple<at::Tensor, at::Tensor> warp2d_backward(const at::Tensor &grad_output, const at::Tensor &input, const at::Tensor &grid,
                                                   int64_t padding, bool align_corners, bool need_input, bool need_grid)
{
    // 16-bit frames, with an fp32 map or one of the frame's type
    const bool half_frames = input.scalar_type() == at::kHalf || input.scalar_type() == at::kBFloat16;
    at::Tensor gin, ggrid;
    // with 16-bit frames the contributions are summed in fp32 and rounded to the frame type once
    if (need_input) gin = at::empty(input.sizes(), half_frames ? input.options().dtype(at::kFloat) : input.options());
    if (need_grid) ggrid = like_layout(grid);
    const pws_tensor dgo = desc(grad_output), din = desc(input), dg = desc(grid);
    pws_tensor dgin, dgg;
    if (need_input) dgin = desc(gin);
    if (need_grid) dgg = desc(ggrid);
    check(pws_warp2d_backward(&dgo, &din, &dg, need_input ? &dgin : nullptr, need_grid ? &dgg : nullptr, PWS_INTERP_BILINEAR, (int)padding,
                              align_corners ? 1 : 0, current_stream(input)));
    if (half_frames && need_input) gin = gin.to(input.scalar_type());
    return std::make_tuple(gin, ggrid);
}

struct WarpFn : public torch::autograd::Function<WarpFn> {
    static at::Tensor forward(torch::autograd::AutogradContext *ctx, const at::Tensor &input, const at::Tensor &grid, int64_t padding,
                              bool align_corners)
    {
        ctx->save_for_backward({input, grid});
        ctx->saved_data["padding"] = padding;
        ctx->saved_data["align_corners"] = align_corners;
        return warp2d_forward(input, grid, padding, align_corners);
    }

    static torch::autograd::variable_list backward(torch::autograd::AutogradContext *ctx, torch::autograd::variable_list grad_outputs)
    {
        const auto saved = ctx->get_saved_variables();
        auto r = warp2d_backward(grad_outputs[0], saved[0], saved[1], ctx->saved_data["padding"].toInt(),
                                 ctx->saved_data["align_corners"].toBool(), ctx->needs_input_grad(0), ctx->needs_input_grad(1));
        return {std::get<0>(r), std::get<1>(r), at::Tensor(), at::Tensor()};
    }
};

// arguments already validated by functional.grid_sample (strings, devices, dimensions, dtypes)
at::Tensor grid_sample(const at::Tensor &input, const at::Tensor &grid, int64_t padding, bool align_corners)
{
    return WarpFn::apply(input, grid, padding, align_corners);
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m)
{
    m.doc() = "compiled PyTorch shim over libpwswarp.so (include/pwswarp.h)";
    m.def("grid_sample", &grid_sample, "forward with an autograd node (bilinear; padding 0 zeros / 1 border)");
    m.def("warp2d_forward", &warp2d_forward, "aten::grid_sampler_2d replacement");
    m.def("warp2d_backward", &warp2d_backward, "aten::grid_sampler_2d_backward replacement -> (grad_input | undefined, grad_grid | undefined)");
    m.def("abi_version", []() { return pws_abi_version(); });
}
