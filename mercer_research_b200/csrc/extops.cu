// extops.cu -- EXTENSIONS (not in the reference): NHWC pooling forward / backward and the softmax + cross-entropy
// epilogue (SURVEY.md section 8a rows x2, x3).
//
// rcn only has max pooling forward on single maps (Pool2D::pool_2d, rcn/src/utils/kernel.rs:245-349; Average panics
// "Not implemented", kernel.rs:283-285) and a sigmoid output layer with quadratic cost (rcn/src/rcn.rs:113,299).
// These kernels complete that family with the reference's own conventions: 2x2 window, stride 2, Same = one zero
// row / column appended at the bottom / right for odd sizes (kernel.rs:253-261), None = trailing row / column
// dropped; window order [(0,0),(0,1),(1,0),(1,1)] with the LAST maximal element winning (kernel.rs:273-281); the
// argmax byte is 2*dy+dx.  Average divides by 4 always.  All are HBM-bound element-wise kernels: one thread per
// output element with the channel index fastest, so every warp access is a contiguous run.  Checked against
// oracle/ext_oracle.cpp ("parity unpinned").
#include "conv.cuh"
#include "dense.cuh"
#include "opctx.cuh"

namespace rcn {

__global__ void __launch_bounds__(256) ext_pool_forward_kernel(const double* __restrict__ x, int H, int W, int C, int Ho, int Wo,
                                                               size_t n_out, int pooling, double* __restrict__ y,
                                                               uint8_t* __restrict__ argmax, int* __restrict__ nan_flag) {
    for (size_t o = blockIdx.x * (size_t)blockDim.x + threadIdx.x; o < n_out; o += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(o % C);
        size_t r = o / C;
        const int ox = (int)(r % Wo); r /= Wo;
        const int oy = (int)(r % Ho);
        const size_t b = r / Ho;
        double p[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int iy = 2 * oy + (i >> 1), ix = 2 * ox + (i & 1);
            p[i] = (iy < H && ix < W) ? x[((b * H + iy) * W + ix) * C + c] : 0.0;
        }
        if (pooling == RCN_POOLING_MAX) {
            int best = 0;
            bool nan = p[0] != p[0];
#pragma unroll
            for (int i = 1; i < 4; ++i) {
                nan = nan || (p[i] != p[i]);
                if (!(p[i] < p[best])) best = i;   // last maximal element wins
            }
            if (nan) *nan_flag = 1;               // partial_cmp(..).unwrap() would panic (kernel.rs:280)
            y[o] = p[best];
            if (argmax) argmax[o] = (uint8_t)best;
        } else {
            y[o] = (((p[0] + p[1]) + p[2]) + p[3]) * 0.25;
        }
    }
}

// One thread per INPUT element: gathers from the single window that covers it (no atomics, every dx written once).
__global__ void __launch_bounds__(256) ext_pool_backward_kernel(const double* __restrict__ dy, const uint8_t* __restrict__ argmax,
                                                                int H, int W, int C, int Ho, int Wo, size_t n_in, int pooling,
                                                                double* __restrict__ dx) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_in; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        size_t r = i / C;
        const int ix = (int)(r % W); r /= W;
        const int iy = (int)(r % H);
        const size_t b = r / H;
        const int oy = iy >> 1, ox = ix >> 1;
        double v = 0.0;
        if (oy < Ho && ox < Wo) {      // None padding: the trailing row / column belongs to no window
            const size_t o = ((b * Ho + oy) * Wo + ox) * C + c;
            const int slot = 2 * (iy & 1) + (ix & 1);
            if (pooling == RCN_POOLING_MAX) v = (argmax[o] == slot) ? dy[o] : 0.0;
            else v = dy[o] * 0.25;
        }
        dx[i] = v;
    }
}

// softmax + cross-entropy over column-major logits (n x B): one warp per sample, lanes stride the classes; the
// max / sum reductions are warp shuffles in a fixed order (deterministic).  The per-sample arithmetic is
// softmax_xent_warp (dense.cuh), which the network's softmax head runs too.
__global__ void __launch_bounds__(256) ext_softmax_xent_kernel(const double* __restrict__ z, int n, size_t B,
                                                               const double* __restrict__ onehot, const int64_t* __restrict__ labels,
                                                               double* __restrict__ probs, double* __restrict__ loss,
                                                               double* __restrict__ delta) {
    const int lane = threadIdx.x & 31;
    const size_t warp = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t b = warp; b < B; b += n_warps) {
        const auto target = [&](int i) { return onehot ? onehot[b * n + i] : ((labels[b] == (int64_t)i) ? 1.0 : 0.0); };
        const auto visit = [&](int i, double, double, double p, double d) {
            if (probs) probs[b * n + i] = p;
            if (delta) delta[b * n + i] = d;
        };
        const double l = softmax_xent_warp(z + b * n, n, lane, target, visit);
        if (loss && lane == 0) loss[b] = l;
    }
}

int pool2d_shape(size_t H, size_t W, int padding, int pooling, size_t* Ho, size_t* Wo) {
    if (padding != RCN_PADDING_NONE && padding != RCN_PADDING_SAME) return fail(RCN_ERR_INVALID, "unknown padding %d", padding);
    if (pooling != RCN_POOLING_AVERAGE && pooling != RCN_POOLING_MAX) return fail(RCN_ERR_INVALID, "unknown pooling %d", pooling);
    if (H < 2 || W < 2)  // kernel.rs:246-251
        return fail(RCN_ERR_SHAPE, "stride_2d expected a matrix with dimensions greater than (2, 2), got (%zu, %zu)", H, W);
    if (H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "map too large");
    const bool same = padding == RCN_PADDING_SAME;
    *Ho = same ? (H + 1) / 2 : H / 2;
    *Wo = same ? (W + 1) / 2 : W / 2;
    return RCN_OK;
}
namespace {
unsigned ew_grid(size_t n) {
    unsigned g = cdiv(n, 256);
    return g > kNumSMs * 16 ? kNumSMs * 16 : (g ? g : 1);
}
}  // namespace

int launch_pool2d_forward(const double* x, size_t B, size_t H, size_t W, size_t C, size_t Ho, size_t Wo, int pooling, double* y,
                          uint8_t* argmax, int* nan_flag, cudaStream_t stream) {
    const size_t n_out = B * Ho * Wo * C;
    if (n_out == 0) return RCN_OK;
    RCN_LAUNCH("ext_pool_forward_kernel", stream,
               ext_pool_forward_kernel<<<ew_grid(n_out), 256, 0, stream>>>(x, (int)H, (int)W, (int)C, (int)Ho, (int)Wo, n_out, pooling,
                                                                           y, argmax, nan_flag));
    return RCN_OK;
}

int launch_pool2d_backward(const double* dy, const uint8_t* argmax, size_t B, size_t H, size_t W, size_t C, size_t Ho, size_t Wo,
                           int pooling, double* dx, cudaStream_t stream) {
    const size_t n_in = B * H * W * C;
    if (n_in == 0) return RCN_OK;
    RCN_LAUNCH("ext_pool_backward_kernel", stream,
               ext_pool_backward_kernel<<<ew_grid(n_in), 256, 0, stream>>>(dy, argmax, (int)H, (int)W, (int)C, (int)Ho, (int)Wo, n_in,
                                                                           pooling, dx));
    return RCN_OK;
}

}  // namespace rcn

using namespace rcn;

extern "C" {

int rcn_cuda_ext_pool2d_forward(int device, void* cuda_stream, const double* x, size_t B, size_t H, size_t W, size_t C,
                                int padding, int pooling, double* y, uint8_t* argmax_out) {
    if (!x || !y) return fail(RCN_ERR_INVALID, "null pointer");
    size_t Ho = 0, Wo = 0;
    RCN_TRY(pool2d_shape(H, W, padding, pooling, &Ho, &Wo));
    const size_t n_out = B * Ho * Wo * C;
    if (n_out == 0) return RCN_OK;
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void* x_dev = nullptr; void* y_dev = nullptr; bool host = false;
    RCN_TRY(c.in(x, B * H * W * C * 8, tl_op_in, &x_dev));
    RCN_TRY(c.out(y, n_out * 8, tl_op_out, &y_dev, &host));
    RCN_TRY(tl_op_aux.reserve(16 + n_out));
    int* flag = tl_op_aux.as<int>();
    RCN_CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), c.stream));
    uint8_t* am_dev = nullptr;
    bool am_host = false;
    if (argmax_out && pooling == RCN_POOLING_MAX) {
        if (is_device_ptr(argmax_out)) am_dev = argmax_out;
        else { am_dev = tl_op_aux.as<uint8_t>() + 16; am_host = true; }
    }
    RCN_TRY(launch_pool2d_forward((const double*)x_dev, B, H, W, C, Ho, Wo, pooling, (double*)y_dev, am_dev, flag, c.stream));
    int nan = 0;
    RCN_CUDA_TRY(cudaMemcpyAsync(&nan, flag, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    if (am_host) RCN_CUDA_TRY(cudaMemcpyAsync(argmax_out, am_dev, n_out, cudaMemcpyDeviceToHost, c.stream));
    if (host) RCN_CUDA_TRY(cudaMemcpyAsync(y, y_dev, n_out * 8, cudaMemcpyDeviceToHost, c.stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(c.stream));
    if (nan) return fail(RCN_ERR_NAN, "called `Option::unwrap()` on a `None` value (partial_cmp on NaN, kernel.rs:280)");
    return RCN_OK;
}

int rcn_cuda_ext_pool2d_backward(int device, void* cuda_stream, const double* dy, const uint8_t* argmax, size_t B, size_t H,
                                 size_t W, size_t C, int padding, int pooling, double* dx) {
    if (!dy || !dx) return fail(RCN_ERR_INVALID, "null pointer");
    size_t Ho = 0, Wo = 0;
    RCN_TRY(pool2d_shape(H, W, padding, pooling, &Ho, &Wo));
    if (pooling == RCN_POOLING_MAX && !argmax) return fail(RCN_ERR_INVALID, "max-pool backward needs the forward pass's argmax");
    const size_t n_in = B * H * W * C, n_out = B * Ho * Wo * C;
    if (n_in == 0) return RCN_OK;
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *dy_dev = nullptr, *am_dev = nullptr; void* dx_dev = nullptr; bool host = false;
    RCN_TRY(c.in(dy, n_out * 8, tl_op_in, &dy_dev));
    if (pooling == RCN_POOLING_MAX) RCN_TRY(c.in(argmax, n_out, tl_op_in2, &am_dev));
    RCN_TRY(c.out(dx, n_in * 8, tl_op_out, &dx_dev, &host));
    RCN_TRY(launch_pool2d_backward((const double*)dy_dev, (const uint8_t*)am_dev, B, H, W, C, Ho, Wo, pooling, (double*)dx_dev,
                                   c.stream));
    return c.finish(dx, dx_dev, n_in * 8, host);
}

int rcn_cuda_ext_softmax_xent(int device, void* cuda_stream, const double* z, size_t n, size_t B, const double* onehot,
                              const int64_t* labels, double* probs, double* loss, double* delta) {
    if (n == 0 || B == 0) return RCN_OK;
    if (!z) return fail(RCN_ERR_INVALID, "null logits");
    if ((onehot == nullptr) == (labels == nullptr)) return fail(RCN_ERR_INVALID, "exactly one of onehot / labels must be given");
    if (n > 0x7fffffff) return fail(RCN_ERR_INVALID, "too many classes");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void *z_dev = nullptr, *t_dev = nullptr; void *p_dev = nullptr, *l_dev = nullptr, *d_dev = nullptr;
    bool hp = false, hl = false, hd = false;
    RCN_TRY(c.in(z, n * B * 8, tl_op_in, &z_dev));
    if (onehot) RCN_TRY(c.in(onehot, n * B * 8, tl_op_in2, &t_dev));
    else RCN_TRY(c.in(labels, B * 8, tl_op_in2, &t_dev));
    if (probs) RCN_TRY(c.out(probs, n * B * 8, tl_op_out, &p_dev, &hp));
    if (loss) RCN_TRY(c.out(loss, B * 8, tl_op_out2, &l_dev, &hl));
    if (delta) RCN_TRY(c.out(delta, n * B * 8, tl_op_ws, &d_dev, &hd));
    unsigned grid = cdiv(B, 8);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("ext_softmax_xent_kernel", c.stream,
               ext_softmax_xent_kernel<<<grid, 256, 0, c.stream>>>((const double*)z_dev, (int)n, B, onehot ? (const double*)t_dev : nullptr,
                                                                   onehot ? nullptr : (const int64_t*)t_dev, (double*)p_dev,
                                                                   (double*)l_dev, (double*)d_dev));
    if (hp) RCN_CUDA_TRY(cudaMemcpyAsync(probs, p_dev, n * B * 8, cudaMemcpyDeviceToHost, c.stream));
    if (hl) RCN_CUDA_TRY(cudaMemcpyAsync(loss, l_dev, B * 8, cudaMemcpyDeviceToHost, c.stream));
    if (hd) RCN_CUDA_TRY(cudaMemcpyAsync(delta, d_dev, n * B * 8, cudaMemcpyDeviceToHost, c.stream));
    if (hp || hl || hd) RCN_CUDA_TRY(cudaStreamSynchronize(c.stream));
    return RCN_OK;
}

}  // extern "C"
