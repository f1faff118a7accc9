// optim.cu -- momentum SGD and AdamW for the convolutional network handle (cnn.cu); the formulas and their operation
// order are in rcn_cuda.h.  Plain SGD (momentum = weight decay = 0) stays on sgd_update_kernel and never comes here.
//
// One launch per step covers the handle's two parameter segments: the conv parameters (gradients [0, n_conv)) and the
// dense model's (gradients [n_conv, n)).  The optimizer state is one flat buffer with the gradient buffer's layout (AdamW:
// m, then v, then t, beta1^t, beta2^t).  Every operation is rounded on its own (__dmul_rn / __dadd_rn / __ddiv_rn /
// __dsqrt_rn: no FMA contraction), so a restatement in numpy reproduces the update bit for bit.  The kernels are memory
// bound (momentum SGD moves 40 B per parameter, AdamW 56 B): 16-byte accesses where every pointer of a segment allows them,
// and a grid-stride loop sized like launch_sgd_update.  In epoch mode block 0 advances the cursor as sgd_update_kernel does.
#include <cmath>

#include "optim.cuh"

namespace rcn {

namespace {

struct OptSeg {
    double* p;
    const double* g;
    double* s0;      // SGD: v; AdamW: m
    double* s1;      // AdamW: v
    size_t n;
    size_t units;    // vec: pairs (the last one may be a single element); otherwise elements
    int vec;
};

template <bool MOMENTUM, bool NESTEROV>
struct SgdOp {
    double B, lambda, mu, eta;
    __device__ __forceinline__ void operator()(double& p, double g, double& v, double&) const {
        const double d = __dadd_rn(__ddiv_rn(g, B), __dmul_rn(lambda, p));
        double u = d;
        if (MOMENTUM) {
            v = __dadd_rn(__dmul_rn(mu, v), d);
            u = NESTEROV ? __dadd_rn(d, __dmul_rn(mu, v)) : v;
        }
        p = __dsub_rn(p, __dmul_rn(eta, u));
    }
};

struct AdamHyper {
    double B, decay, b1, omb1, b2, omb2, eps, eta;
};

struct AdamOp {
    AdamHyper h;
    double c1, c2;   // 1 - beta1^t, 1 - beta2^t of this step
    __device__ __forceinline__ void operator()(double& p, double g, double& m, double& v) const {
        p = __dmul_rn(p, h.decay);
        const double gh = __ddiv_rn(g, h.B);
        m = __dadd_rn(__dmul_rn(h.b1, m), __dmul_rn(h.omb1, gh));
        v = __dadd_rn(__dmul_rn(h.b2, v), __dmul_rn(h.omb2, __dmul_rn(gh, gh)));
        const double den = __dadd_rn(__dsqrt_rn(__ddiv_rn(v, c2)), h.eps);
        p = __dsub_rn(p, __dmul_rn(h.eta, __ddiv_rn(__ddiv_rn(m, c1), den)));
    }
};

// NS: state arrays per parameter (0: SGD without momentum, 1: SGD with momentum, 2: AdamW)
template <int NS, class Op>
__device__ __forceinline__ void optim_segment(const OptSeg& s, size_t j, size_t stride, const Op& op) {
    for (; j < s.units; j += stride) {
        if (s.vec && 2 * j + 1 < s.n) {
            double2 p = reinterpret_cast<const double2*>(s.p)[j];
            const double2 g = __ldg(reinterpret_cast<const double2*>(s.g) + j);
            double2 a = make_double2(0.0, 0.0), b = a;
            if (NS > 0) a = reinterpret_cast<const double2*>(s.s0)[j];
            if (NS > 1) b = reinterpret_cast<const double2*>(s.s1)[j];
            op(p.x, g.x, a.x, b.x);
            op(p.y, g.y, a.y, b.y);
            reinterpret_cast<double2*>(s.p)[j] = p;
            if (NS > 0) reinterpret_cast<double2*>(s.s0)[j] = a;
            if (NS > 1) reinterpret_cast<double2*>(s.s1)[j] = b;
        } else {
            const size_t i = s.vec ? 2 * j : j;
            double p = s.p[i], a = 0.0, b = 0.0;
            if (NS > 0) a = s.s0[i];
            if (NS > 1) b = s.s1[i];
            op(p, __ldg(s.g + i), a, b);
            s.p[i] = p;
            if (NS > 0) s.s0[i] = a;
            if (NS > 1) s.s1[i] = b;
        }
    }
}

template <int NS, class Op>
__device__ __forceinline__ void optim_body(const OptSeg& a, const OptSeg& b, const Op& op, long long* cursor, long long batch,
                                           long long n_samples) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    optim_segment<NS>(a, t, stride, op);
    // segment b continues the grid-stride sweep where segment a ended, so the threads share both evenly
    optim_segment<NS>(b, (t + stride - a.units % stride) % stride, stride, op);
    if (cursor && blockIdx.x == 0 && threadIdx.x == 0) {
        // next chunk of training_set.chunks_exact(batch) (rcn.rs:147); the remainder is dropped, then wrap
        long long c = *cursor + batch;
        if (c + batch > n_samples) c = 0;
        *cursor = c;
    }
}

template <bool MOMENTUM, bool NESTEROV>
__global__ void __launch_bounds__(256) optim_sgd_kernel(OptSeg a, OptSeg b, SgdOp<MOMENTUM, NESTEROV> op,
                                                        long long* __restrict__ cursor, long long batch, long long n_samples) {
    optim_body<MOMENTUM ? 1 : 0>(a, b, op, cursor, batch, n_samples);
}

// scal = {t, beta1^t, beta2^t}.  Every CTA reads them before it takes its ticket; the last CTA to take one has therefore
// seen every read and alone writes the advanced values, then resets the ticket for the next launch (graph replay).
__global__ void __launch_bounds__(256) optim_adamw_kernel(OptSeg a, OptSeg b, AdamHyper h, double* __restrict__ scal,
                                                          unsigned* __restrict__ ticket, long long* __restrict__ cursor,
                                                          long long batch, long long n_samples) {
    __shared__ double s_sc[3];
    if (threadIdx.x < 3) s_sc[threadIdx.x] = __ldcg(scal + threadIdx.x);
    __syncthreads();
    const double b1t = __dmul_rn(s_sc[1], h.b1), b2t = __dmul_rn(s_sc[2], h.b2);
    const AdamOp op{h, __dsub_rn(1.0, b1t), __dsub_rn(1.0, b2t)};
    optim_body<2>(a, b, op, cursor, batch, n_samples);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
            *ticket = 0;
            scal[0] = __dadd_rn(s_sc[0], 1.0);
            scal[1] = b1t;
            scal[2] = b2t;
        }
    }
}

bool in_unit(double x) { return std::isfinite(x) && x >= 0.0 && x < 1.0; }

OptSeg make_seg(double* p, const double* g, double* s0, double* s1, size_t n) {
    const uintptr_t align = (uintptr_t)p | (uintptr_t)g | (uintptr_t)s0 | (uintptr_t)s1;
    OptSeg s{p, g, s0, s1, n, n, align % 16 == 0 ? 1 : 0};
    if (s.vec) s.units = (n + 1) / 2;
    return s;
}

}  // namespace

int optim_validate(const OptimConfig& c) {
    if (c.kind == RCN_OPTIMIZER_SGD) {
        if (!in_unit(c.momentum)) return fail(RCN_ERR_INVALID, "SGD momentum %g is outside [0, 1)", c.momentum);
        if (c.nesterov != 0 && c.nesterov != 1) return fail(RCN_ERR_INVALID, "nesterov must be 0 or 1, got %d", c.nesterov);
        if (c.nesterov && c.momentum == 0.0) return fail(RCN_ERR_INVALID, "Nesterov momentum needs momentum > 0");
    } else if (c.kind == RCN_OPTIMIZER_ADAMW) {
        if (!in_unit(c.beta1) || !in_unit(c.beta2))
            return fail(RCN_ERR_INVALID, "AdamW betas (%g, %g) must lie in [0, 1)", c.beta1, c.beta2);
        if (!(std::isfinite(c.eps) && c.eps > 0.0)) return fail(RCN_ERR_INVALID, "AdamW eps %g must be finite and > 0", c.eps);
    } else {
        return fail(RCN_ERR_INVALID, "unknown optimizer %d", c.kind);
    }
    if (!(std::isfinite(c.weight_decay) && c.weight_decay >= 0.0))
        return fail(RCN_ERR_INVALID, "weight decay %g must be finite and >= 0", c.weight_decay);
    return RCN_OK;
}

size_t optim_state_len(const OptimConfig& c, size_t n) {
    if (c.kind == RCN_OPTIMIZER_ADAMW) return 2 * n + 3;
    return c.momentum > 0.0 ? n : 0;
}

int optim_reset_state(const OptimConfig& c, double* state, size_t n, cudaStream_t stream) {
    const size_t len = optim_state_len(c, n);
    if (len == 0) return RCN_OK;
    RCN_CUDA_TRY(cudaMemsetAsync(state, 0, len * sizeof(double), stream));
    if (c.kind == RCN_OPTIMIZER_ADAMW) {
        static const double start[3] = {0.0, 1.0, 1.0};   // t, beta1^t, beta2^t
        RCN_CUDA_TRY(cudaMemcpyAsync(state + 2 * n, start, sizeof(start), cudaMemcpyHostToDevice, stream));
    }
    return RCN_OK;
}

int launch_optim_update(const OptimConfig& c, double* p0, size_t n0, double* p1, size_t n1, const double* g, double* state,
                        unsigned* ticket, double eta, size_t global_batch, cudaStream_t stream, long long* cursor,
                        long long batch, long long n_samples) {
    if (n0 + n1 == 0 && !cursor) return RCN_OK;
    const size_t n = n0 + n1;
    const bool adam = c.kind == RCN_OPTIMIZER_ADAMW;
    const bool mom = !adam && c.momentum > 0.0;
    double* m = (adam || mom) ? state : nullptr;
    double* v = adam ? state + n : nullptr;
    const OptSeg a = make_seg(p0, g, m, v, n0);
    const OptSeg b = make_seg(p1, g + n0, m ? m + n0 : nullptr, v ? v + n0 : nullptr, n1);
    const size_t units = a.units + b.units;
    unsigned grid = units ? cdiv(units, 256) : 1;   // no parameters with a cursor: only the cursor advances
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    const double B = (double)global_batch;
    if (adam) {
        // (1 - eta * lambda), (1 - beta1), (1 - beta2) formed here, once
        const AdamHyper h{B, 1.0 - eta * c.weight_decay, c.beta1, 1.0 - c.beta1, c.beta2, 1.0 - c.beta2, c.eps, eta};
        RCN_LAUNCH("optim_adamw_kernel", stream,
                   optim_adamw_kernel<<<grid, 256, 0, stream>>>(a, b, h, state + 2 * n, ticket, cursor, batch, n_samples));
        return RCN_OK;
    }
#define RCN_OPTIM_SGD(M, N)                                                                                              \
    RCN_LAUNCH("optim_sgd_kernel", stream,                                                                               \
               (optim_sgd_kernel<M, N><<<grid, 256, 0, stream>>>(a, b, SgdOp<M, N>{B, c.weight_decay, c.momentum, eta}, cursor, \
                                                                  batch, n_samples)))
    if (!mom) RCN_OPTIM_SGD(false, false);
    else if (c.nesterov) RCN_OPTIM_SGD(true, true);
    else RCN_OPTIM_SGD(true, false);
#undef RCN_OPTIM_SGD
    return RCN_OK;
}

}  // namespace rcn
