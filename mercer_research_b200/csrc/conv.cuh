// conv.cuh -- launch entry points of the learned-convolution, pooling and activation kernels (conv.cu, extops.cu),
// shared by the op-level extensions and the convolutional network handle (cnn.cu).
#pragma once
#include "common.cuh"

namespace rcn {

struct OzakiWorkspace;

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SIGMOID = 2 };

struct ConvShape {
    size_t B, H, W, Ci, Co, kh, kw;
    int padding;
    size_t Ho = 0, Wo = 0;
    int ph, pw;
};

// The convolve_2d contract (kernel.rs:123-135) extended to channels: status codes and messages of the ext ops.
int check_conv_shape(size_t B, size_t H, size_t W, size_t Ci, size_t Co, size_t kh, size_t kw, int padding, ConvShape* s);
// Does the forward pass of `s` take the direct small-channel kernel?
bool conv_direct_ok(const ConvShape& s);

// `tw` / `rs`: the tcgen05 workspace and the bias-gradient reduction scratch; NULL = this thread's per-device ones.
int launch_conv2d_forward(const double* x, const double* w, const double* bias, const ConvShape& s, int act, double* y,
                          cudaStream_t stream, OzakiWorkspace* tw = nullptr);
// The direct kernel reading u8 pixels (one channel, Ci == 1); requires conv_direct_ok(s).
int launch_conv2d_forward_u8(const uint8_t* x, const double* w, const double* bias, const ConvShape& s, int act, double* y,
                             cudaStream_t stream);
int launch_conv2d_backward_data(const double* dz, const double* w, const ConvShape& s, const double* y_prev, int act_prev,
                                double* dx, DevBuf& ws, cudaStream_t stream, OzakiWorkspace* tw = nullptr);
int launch_conv2d_backward_weight(const double* x, const double* dz, const ConvShape& s, double* dw, double* db, DevBuf& ws,
                                  cudaStream_t stream, OzakiWorkspace* tw = nullptr, ReduceScratch* rs = nullptr);
// dz = dy .* act'(y), act' from the stored output y
int launch_activation_backward(const double* y, const double* dy, size_t n, int act, double* dz, cudaStream_t stream);

// Pool2D contract (kernel.rs:246-251) on an H x W map; the pooled size goes to Ho, Wo.
int pool2d_shape(size_t H, size_t W, int padding, int pooling, size_t* Ho, size_t* Wo);
// NHWC 2x2 / stride-2 pooling; argmax (max only, may be NULL); nan_flag set to 1 when a max window holds a NaN.
int launch_pool2d_forward(const double* x, size_t B, size_t H, size_t W, size_t C, size_t Ho, size_t Wo, int pooling, double* y,
                          uint8_t* argmax, int* nan_flag, cudaStream_t stream);
int launch_pool2d_backward(const double* dy, const uint8_t* argmax, size_t B, size_t H, size_t W, size_t C, size_t Ho, size_t Wo,
                           int pooling, double* dx, cudaStream_t stream);

}  // namespace rcn
