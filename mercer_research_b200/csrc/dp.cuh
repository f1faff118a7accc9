// dp.cuh -- data-parallel gradient exchange fused with the SGD update, over NVLink peer memory (see dp.cu).
#pragma once
#include "common.cuh"
#include "timeline.cuh"

namespace rcn {

constexpr int kDpMaxWorld = 16;
constexpr int kDpThreads = 1024;   // threads per CTA of the exchange kernel
constexpr int kDpMaxCtas = 20;     // its grid: few, fat CTAs so that the next step's kernels find their SMs free beside it (dp.cu)

// One rank's communication block (device memory, exported to the peers):
//   [ctrl: step | done_ctas | pad to 256 B][receive slots: 2 (step parity) x world x n doubles, sentinel-filled]
struct DpState {
    bool connected = false;
    int world = 1, rank = 0;
    size_t n = 0, bytes = 0;
    void* block = nullptr;                 // this rank's block
    void* peers[kDpMaxWorld] = {};         // every rank's block as mapped into THIS process (peers[rank] == block)
    bool imported[kDpMaxWorld] = {};       // mapped with cudaIpcOpenMemHandle (must be closed)
};

// Handed to a gradient-producing kernel so that it can PUSH its final gradient values into the peers' receive slots
// itself (the exchange then overlaps that kernel's tail and the next launch); world == 1 means "do not push".
// Always passed as a `__grid_constant__` kernel parameter: the peer table is then indexed in the constant bank instead of
// being copied to a per-thread stack frame.
struct DpPush {
    char* peers[kDpMaxWorld];
    int world, rank;
    unsigned long long n;
    unsigned long long timeout_ns;   // bound on one receive's wait (RCN_CUDA_DP_TIMEOUT_MS, default 10 s)
    Timeline* tl;                    // device-side launch timeline of the exchange kernel (timeline.cuh), null = off
};
DpPush dp_push_desc(const DpState& st);
constexpr size_t kDpCtrlBytesPub = 256;   // offset of the receive slots inside a communication block

// Control words at the head of a communication block.
struct DpCtrl {
    long long step;              // exchanges completed by this rank (device-side: CUDA-graph replayable)
    unsigned int done_ctas;      // ticket of the kernel that is finishing the current exchange
    unsigned int error;          // sticky: a receive timed out (a peer never pushed); read back by rcn_cuda_dp_error
};
constexpr unsigned long long kDpSentinelBits = 0xFFFFFFFFFFFFFFFFull;
constexpr unsigned long long kDpQuietNaNBits = 0x7FF8000000000000ull;

#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long dp_ld_volatile(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// Device side of the push: slot [step parity][my rank][i] on every peer = v (the sentinel itself is never sent).
__device__ __forceinline__ void dp_push_value(const DpPush& dp, size_t par_off, size_t i, double v) {
    unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    if (bits == kDpSentinelBits) bits = kDpQuietNaNBits;
    for (int q = 0; q < dp.world; ++q)
        if (q != dp.rank)
            reinterpret_cast<unsigned long long*>(dp.peers[q] + kDpCtrlBytesPub)[par_off + (size_t)dp.rank * dp.n + i] = bits;
}

// Slow path of a receive: the peer's value has not arrived yet.  Polls with a BOUND: every 1024 polls the thread looks at
// the sticky error word and at %globaltimer; when a peer stays silent for timeout_ns (it died, raised before its launch, or
// runs a different number of steps) the error word is set and NaN is returned, so the step finishes with NaN parameters
// and rcn_cuda_dp_error / the next host call reports the broken group instead of the device hanging in this loop.
static __device__ __noinline__ unsigned long long dp_wait_slot(const unsigned long long* p, DpCtrl* ctrl, unsigned long long timeout_ns) {
    unsigned long long t0 = 0;
    for (unsigned spins = 1;; ++spins) {
        const unsigned long long bits = dp_ld_volatile(p);
        if (bits != kDpSentinelBits) return bits;
        if ((spins & 1023u) == 0) {
            if (*reinterpret_cast<volatile unsigned int*>(&ctrl->error)) return kDpQuietNaNBits;
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (!t0) t0 = t;
            else if (t - t0 > timeout_ns) { atomicExch(&ctrl->error, 1u); return kDpQuietNaNBits; }
        }
    }
}

// Device side of the receive for ONE element: every peer's value of element i in my own block is REQUESTED first (one L2
// round trip for all of them, not world - 1 dependent ones), then those still holding the sentinel are polled; the sentinel
// is put back and the ranks are added in RANK ORDER (mine = `own`), so every replica computes the bit-identical global sum.
// WORLD = 0: runtime world size (groups of 8).
template <int WORLD>
__device__ __forceinline__ double dp_receive_sum(const DpPush& dp, size_t par_off, size_t i, double own) {
    unsigned long long* slots = reinterpret_cast<unsigned long long*>(dp.peers[dp.rank] + kDpCtrlBytesPub) + par_off + i;
    DpCtrl* ctrl = reinterpret_cast<DpCtrl*>(dp.peers[dp.rank]);
    const int world = WORLD ? WORLD : dp.world;
    constexpr int G = WORLD ? WORLD : 8;
    double s = 0.0;
    for (int q0 = 0; q0 < world; q0 += G) {
        unsigned long long b[G];
#pragma unroll
        for (int u = 0; u < G; ++u) {
            const int q = q0 + u;
            b[u] = 0;
            if (q < world && q != dp.rank) b[u] = dp_ld_volatile(slots + (size_t)q * dp.n);
        }
#pragma unroll
        for (int u = 0; u < G; ++u) {
            const int q = q0 + u;
            if (q < world) {
                double v = own;
                if (q != dp.rank) {
                    unsigned long long* p = slots + (size_t)q * dp.n;
                    if (b[u] == kDpSentinelBits) b[u] = dp_wait_slot(p, ctrl, dp.timeout_ns);
                    *p = kDpSentinelBits;
                    v = __longlong_as_double((long long)b[u]);
                }
                s = (q == 0) ? v : s + v;
            }
        }
    }
    return s;
}

// parity offset of the step this rank is about to exchange (reads the device-side step counter of its own block)
__device__ __forceinline__ size_t dp_push_parity_offset(const DpPush& dp) {
    const long long step = *reinterpret_cast<volatile long long*>(dp.peers[dp.rank]) + 1;
    return (size_t)(step & 1) * dp.world * dp.n;
}
#endif

size_t dp_block_bytes(int world, size_t n);
int dp_alloc(DpState& st, int world, int rank, size_t n, cudaStream_t stream);
void dp_release(DpState& st);
// Reads the sticky error word of this rank's block (synchronises `stream` first): non-zero = a receive timed out.
int dp_read_error(const DpState& st, cudaStream_t stream, unsigned* error);

// params[i] -= scale * sum_r grads_r[i], r ascending, identical on every rank; grads[i] <- the global sum.
// cursor / batch / n_samples: optional epoch cursor advanced like sgd_update_kernel does.
// already_pushed: the gradient kernel pushed this step's values itself (DpPush); the kernel then only receives.
int launch_dp_allreduce_sgd(const DpState& st, double* params, double* grads, double scale, cudaStream_t stream,
                            long long* cursor, long long batch, long long n_samples, const double* stats = nullptr,
                            double* stats_ring = nullptr, bool already_pushed = false, Timeline* tl = nullptr);

}  // namespace rcn
