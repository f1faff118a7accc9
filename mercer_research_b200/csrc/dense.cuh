// dense.cuh -- fully-connected layer kernels (f64): forward, backward-data, backward-weight, SGD step.
// Reference: rcn/src/rcn.rs:105-116 (classify_test), :260-314 (backprop), :176-223 (train_batch).
#pragma once
#include "common.cuh"

namespace rcn {

struct OzakiWorkspace;   // ozaki.cuh: scratch of the tcgen05 integer-slice GEMM (NULL = never take that path)

// env RCN_CUDA_GEMM: (unset) auto = tcgen05 integer slices for large dense layers, DMMA otherwise; "dmma"; "tc" forces the
// tcgen05 path for every GEMM; "simt" selects the plain SIMT cross-check kernels.
enum GemmImpl { GEMM_AUTO = 0, GEMM_DMMA = 1, GEMM_SIMT = 2, GEMM_TC = 3 };
GemmImpl gemm_impl();

// A_out (M x N) = sigmoid(W (M x K) * A_in (K x N) + b 1^T)                         rcn.rs:113 / :287-289
// If delta_out != NULL (last layer): delta_out = (A_out - Y) .* A_out .* (1 - A_out)  rcn.rs:299
//   with Y given either as one-hot matrix (M x N) or as labels (N).
int launch_dense_forward(const double* W, const double* b, const double* A_in, size_t M, size_t K, size_t N,
                         double* A_out, double* delta_out, const double* onehot, const int64_t* labels,
                         cudaStream_t stream, OzakiWorkspace* oz = nullptr);

// delta_out (M x N) = (W_up^T (M x K) * delta_up (K x N)) .* A (M x N) .* (1 - A)    rcn.rs:305-309
// W_up is stored K x M (rows = upper layer width).
int launch_dense_backward_data(const double* W_up, const double* delta_up, const double* A, size_t M, size_t K,
                               size_t N, double* delta_out, cudaStream_t stream, OzakiWorkspace* oz = nullptr);

// dx (M x N) = W0^T (M x K) * delta0 (K x N): the gradient of the cost with respect to the dense stack's input (no
// activation derivative); W0 is stored K x M.  Same DMMA / tcgen05 choice as launch_dense_backward_data.
int launch_dense_input_grad(const double* W0, const double* delta0, size_t M, size_t K, size_t N, double* dx, cudaStream_t stream,
                            OzakiWorkspace* oz = nullptr);

// dW (M x N) = delta (M x Kb) * A_prev (N x Kb)^T, db (M) = delta * 1                 rcn.rs:302-303,309-310 summed
// over the batch (rcn.rs:190-205).  workspace: split-K partials.
int launch_dense_backward_weight(const double* delta, const double* A_prev, size_t M, size_t N, size_t Kb, double* dW,
                                 double* db, DevBuf& workspace, ReduceScratch& rs, cudaStream_t stream, OzakiWorkspace* oz = nullptr);

// out[i] = sum_p partials[p*n + i], p ascending (deterministic split-K combine)
int launch_reduce_splits(const double* partials, int splits, size_t n, double* out, cudaStream_t stream);
// db[m] = sum_n delta[m + n*M]  (delta M x N column-major), fixed summation order
int launch_bias_grad(const double* delta, size_t M, size_t N, double* db, ReduceScratch& rs, cudaStream_t stream);

// params -= scale * grads   (rcn.rs:210-222, scale = eta / batch formed first)
// cursor (optional): device-side position of the epoch walk, advanced by `batch` with chunks_exact wrap-around (also when
// n == 0: one thread then only advances the cursor).
// stats / stats_ring (optional, with cursor): the step's {cost, hits} pair is copied to stats_ring + 2 * (cursor / batch)
// (pinned host memory in rcn_cuda_train_epoch_host) before the cursor advances.
int launch_sgd_update(double* params, const double* grads, size_t n, double scale, cudaStream_t stream,
                      long long* cursor = nullptr, long long batch = 0, long long n_samples = 0, const double* stats = nullptr,
                      double* stats_ring = nullptr);

// labels[b] = argmax_i acts[i, b], last maximal element wins (rcn.rs:92-97)
int launch_argmax_last(const double* acts, size_t n, size_t B, int64_t* labels, cudaStream_t stream);

// stats[0] = sum_b 0.5*|a_b - y_b|^2 (as double), stats[1] = bit pattern of uint64 hit count (rcn.rs:153-157)
int launch_batch_stats(const double* acts, size_t n, size_t B, const double* onehot, const int64_t* labels,
                       double* stats_dev, ReduceScratch& rs, cudaStream_t stream);

// Z (M x N) = W (M x K) * A_in (K x N) + b 1^T with no activation: the logits of the softmax cross-entropy head, on the
// engine launch_dense_forward would pick for the same shape.
int launch_dense_logits(const double* W, const double* b, const double* A_in, size_t M, size_t K, size_t N, double* Z,
                        cudaStream_t stream, OzakiWorkspace* oz = nullptr);

// Softmax cross-entropy head over the logits z (n x B column-major), in place: z becomes p = softmax(z) per sample.
// delta (optional, training): p - onehot(label).  labels_out (optional): the rcn.rs:92-97 last-max-wins argmax of z.
// stats (optional, needs labels): stats[0] = sum_b of the per-sample cost (log s + m) - z_label, stats[1] = bit pattern of
// the uint64 count of samples whose set {i : z_i = max z} is {label}.  Labels outside [0, n) have an all-zero target.
int launch_softmax_xent_head(double* z, size_t n, size_t B, const int64_t* labels, double* delta, int64_t* labels_out,
                             double* stats_dev, ReduceScratch& rs, cudaStream_t stream);

#ifdef __CUDACC__
// Softmax + cross-entropy of one sample's logits z[0..n) on one warp (lanes stride the classes); the reductions are warp
// shuffles in a fixed order (deterministic): m = max z, then s = sum exp(z - m), then ls = log s.  Then for each of the
// lane's classes i, in ascending order, with y = target(i): p = exp(z_i - m) / s and visit(i, z_i, m, p, p - y), where
// z_i was read before visit is called (so visit may overwrite z in place).  Returns, on every lane, the sample's cost
// sum_i y_i ((ls + m) - z_i) over the classes with y_i != 0.  ext_softmax_xent_kernel and softmax_xent_head_kernel share
// this arithmetic.
template <class Target, class Visit>
__device__ __forceinline__ double softmax_xent_warp(const double* z, int n, int lane, const Target& target, const Visit& visit) {
    double m = -INFINITY;
    for (int i = lane; i < n; i += 32) m = fmax(m, z[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    double s = 0.0;
    for (int i = lane; i < n; i += 32) s += exp(z[i] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double ls = log(s);
    double l = 0.0;
    for (int i = lane; i < n; i += 32) {
        const double y = target(i);
        const double zi = z[i];
        const double p = exp(zi - m) / s;
        visit(i, zi, m, p, p - y);
        if (y != 0.0) l += y * ((ls + m) - zi);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    return l;
}
#endif

}  // namespace rcn
