// optim.cuh -- the convolutional network handle's optimizers other than plain SGD (semantics in rcn_cuda.h).
#pragma once
#include "common.cuh"

namespace rcn {

struct OptimConfig {
    int kind = RCN_OPTIMIZER_SGD;
    double momentum = 0.0;
    int nesterov = 0;
    double weight_decay = 0.0;
    double beta1 = 0.9, beta2 = 0.999, eps = 1e-8;
};

// RCN_ERR_INVALID for an unknown kind or an out-of-range / non-finite hyperparameter of that kind.
int optim_validate(const OptimConfig& c);
// SGD with momentum = weight_decay = 0: the handle keeps its sgd_update_kernel launches and has no state.
inline bool optim_is_plain(const OptimConfig& c) {
    return c.kind == RCN_OPTIMIZER_SGD && c.momentum == 0.0 && c.weight_decay == 0.0;
}
// Length of the exported state for n parameters: SGD with momentum v (n), AdamW m | v | t, beta1^t, beta2^t (2n + 3).
size_t optim_state_len(const OptimConfig& c, size_t n);
// Initial state (state_len doubles, device): zeros, with beta1^t = beta2^t = 1 for AdamW.
int optim_reset_state(const OptimConfig& c, double* state, size_t n, cudaStream_t stream);

// One optimizer step over two parameter segments, p0 (n0) and p1 (n1), whose gradient sums are g[0, n0) and g[n0, n0+n1)
// and whose state has the layout of g.  `ticket`: one zeroed u32 (AdamW), reset by the kernel.  `cursor` (optional)
// advances by `batch` over `n_samples` like sgd_update_kernel's.  One launch, also when n0 + n1 == 0 with a cursor.
int launch_optim_update(const OptimConfig& c, double* p0, size_t n0, double* p1, size_t n1, const double* g, double* state,
                        unsigned* ticket, double eta, size_t global_batch, cudaStream_t stream, long long* cursor = nullptr,
                        long long batch = 0, long long n_samples = 0);

}  // namespace rcn
