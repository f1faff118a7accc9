// dp.cu -- the exchange step of rcn's minibatch gradient sum, scaled from host threads to the GPUs of one box.
//
// Reference: rcn/src/rcn.rs:190-205 sums the per-sample gradients of a minibatch over rayon worker threads behind two
// mutexes, then rcn.rs:210-222 applies W -= (eta/B) * sum.  Data-parallel on N GPUs the same sum runs over ranks:
// every rank holds gradient SUMS of its shard in the flat buffer [dW0|db0|dW1|db1|...], the ranks' buffers are added
// and every replica applies the identical update (SURVEY.md section 8e).
//
// For the latency-bound regime (rcn's canonical 784-30-10 network has 23 860 parameters = 190 KB) a library
// all-reduce costs more than the whole training step, so exchange and update are ONE kernel over NVLink / NVSwitch
// peer memory:
//   * every rank owns a communication block (cudaMalloc, exported to the peers with cudaIpcGetMemHandle or, inside
//     one process, mapped with cudaDeviceEnablePeerAccess) holding 2 x world receive slots of n doubles, pre-filled
//     with a SENTINEL bit pattern (all ones -- a NaN payload no arithmetic produces);
//   * each thread PUSHES its elements of the local gradient into slot [step parity][my rank] of every peer (plain
//     8-byte stores to peer addresses travel over NVLink; an 8-byte store is single-copy atomic, so the value itself
//     is the arrival flag -- the low-latency protocol NCCL calls LL, without a separate flag, fence or barrier);
//   * the same thread then polls its elements of the peers' slots in ITS OWN block until they differ from the sentinel,
//     puts the sentinel back, adds the ranks in RANK ORDER (so all replicas compute bit-identical sums and stay
//     bit-identical to each other) and applies the update.  Latency = one NVLink traversal + a few L2 polls.
// All of a thread's peer slots are requested before any is tested (one L2 round trip, not world - 1 dependent ones) and
// every wait is BOUNDED (dp_wait_slot: a silent peer sets a sticky error word and yields NaN instead of hanging the
// device).  The kernel runs as a FEW FAT CTAs (<= 20 x 1024 threads, grid-stride): beside rcn's canonical step its
// successor, kernel A of the next step (128 CTAs that each need a whole SM), then finds its SMs free and can run its
// parameter-independent front end while this kernel waits for the NVLink traffic (smallnet.cu).
// Threads are independent: no grid-wide, CTA-wide or end-of-kernel barrier.  The receive slots are double buffered by
// step parity: a peer can only push step s+2 into the parity that held step s after it has received every rank's
// step s+1 push, which a rank issues only after its step-s kernel (reads and sentinel resets included) has finished.
// The step counter lives in device memory, so a captured CUDA graph replays the kernel unchanged.  Large gradient
// buffers (e.g. the 268 MB of the 4096-wide MLP) are bandwidth-bound and stay on NCCL (trainer.py picks by size).
#include "dp.cuh"

#include <cstdlib>

namespace rcn {

constexpr size_t kDpCtrlBytes = 256;

size_t dp_block_bytes(int world, size_t n) { return kDpCtrlBytes + 2 * (size_t)world * n * sizeof(double); }

int dp_alloc(DpState& st, int world, int rank, size_t n, cudaStream_t stream) {
    if (world < 1 || world > kDpMaxWorld || rank < 0 || rank >= world) return fail(RCN_ERR_INVALID, "bad world / rank (%d / %d)", world, rank);
    dp_release(st);
    st.world = world; st.rank = rank; st.n = n;
    st.bytes = dp_block_bytes(world, n);
    RCN_CUDA_TRY(cudaMalloc(&st.block, st.bytes));
    alloc_generation().fetch_add(1, std::memory_order_relaxed);   // peer pointers are baked into captured step graphs too
    RCN_CUDA_TRY(cudaMemsetAsync(st.block, 0xFF, st.bytes, stream));      // every receive slot = sentinel
    RCN_CUDA_TRY(cudaMemsetAsync(st.block, 0, kDpCtrlBytes, stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(stream));
    st.peers[rank] = st.block;
    return RCN_OK;
}

void dp_release(DpState& st) {
    for (int q = 0; q < kDpMaxWorld; ++q) {
        if (st.imported[q] && st.peers[q]) cudaIpcCloseMemHandle(st.peers[q]);
        st.peers[q] = nullptr; st.imported[q] = false;
    }
    if (st.block) { cudaFree(st.block); alloc_generation().fetch_add(1, std::memory_order_relaxed); }
    st.block = nullptr; st.connected = false; st.world = 1; st.rank = 0;
    cudaGetLastError();
}

static_assert(kDpCtrlBytes == kDpCtrlBytesPub, "slot offset mismatch");
static_assert(sizeof(DpCtrl) <= kDpCtrlBytes, "control words must fit the block header");

static unsigned long long dp_timeout_ns() {
    static const unsigned long long ns = []() {
        const char* e = getenv("RCN_CUDA_DP_TIMEOUT_MS");
        const long long ms = e ? atoll(e) : 10000;
        return (unsigned long long)(ms > 0 ? ms : 10000) * 1000000ull;
    }();
    return ns;
}

DpPush dp_push_desc(const DpState& st) {
    DpPush d{};
    d.world = st.connected ? st.world : 1;
    d.rank = st.rank;
    d.n = st.n;
    d.timeout_ns = dp_timeout_ns();
    for (int q = 0; q < st.world && q < kDpMaxWorld; ++q) d.peers[q] = (char*)st.peers[q];
    return d;
}

int dp_read_error(const DpState& st, cudaStream_t stream, unsigned* error) {
    *error = 0;
    if (!st.block) return RCN_OK;
    DpCtrl c{};
    RCN_CUDA_TRY(cudaMemcpyAsync(&c, st.block, sizeof(c), cudaMemcpyDeviceToHost, stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(stream));
    *error = c.error;
    return RCN_OK;
}

template <int WORLD>   // 0 = runtime world size
__global__ void __launch_bounds__(kDpThreads, 1) dp_allreduce_sgd_kernel(const __grid_constant__ DpPush dp, double* __restrict__ params,
                                                                          double* __restrict__ grads, double scale,
                                                                          long long* __restrict__ cursor, long long batch,
                                                                          long long n_samples, const double* __restrict__ stats,
                                                                          double* __restrict__ stats_ring, int already_pushed) {
    // programmatic dependent launch (no-ops unless the host asked for it): wait for the gradient kernel to complete, THEN
    // let the next kernel's launch proceed under this one (its pre-wait part may rely on everything up to the gradient
    // kernel being complete, see smallnet.cu)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    RCN_TL_BEGIN(dp.tl, 2);
    DpCtrl* ctrl = reinterpret_cast<DpCtrl*>(dp.peers[dp.rank]);
    const long long step = *reinterpret_cast<volatile long long*>(&ctrl->step) + 1;
    const size_t n = dp.n;
    const size_t par_off = (size_t)(step & 1) * (WORLD ? WORLD : dp.world) * n;
    const size_t stride = (size_t)gridDim.x * kDpThreads;
    const size_t first = (size_t)blockIdx.x * kDpThreads + threadIdx.x;
    // ---- push my elements of the local gradient sums into my slot on every peer (stores travel over NVLink) ---------
    if (!already_pushed)
        for (size_t i = first; i < n; i += stride) dp_push_value(dp, par_off, i, grads[i]);
    // ---- receive: my elements of every peer's slot in my own block, sentinel restored, ranks added in rank order --------
    for (size_t i = first; i < n; i += stride) {
        const double pold = params[i];
        const double s = dp_receive_sum<WORLD>(dp, par_off, i, grads[i]);
        grads[i] = s;                            // the gradient buffer ends up holding the global sum, like an all-reduce
        params[i] = sgd_apply(pold, scale, s);   // W -= (eta / B) * sum   (rcn.rs:214,221)
    }
    // ---- the last CTA to finish advances the device-side step counter (and the epoch cursor) ----------------------------
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int t = atomicAdd(&ctrl->done_ctas, 1u);
        if (t == gridDim.x - 1) {
            ctrl->done_ctas = 0;
            *reinterpret_cast<volatile long long*>(&ctrl->step) = step;
            if (cursor) {
                if (stats_ring) {
                    double* dst = stats_ring + 2 * (*cursor / batch);
                    dst[0] = stats[0];
                    dst[1] = stats[1];
                }
                long long cc = *cursor + batch;
                if (cc + batch > n_samples) cc = 0;
                *cursor = cc;
            }
            __threadfence();
        }
    }
    RCN_TL_END(dp.tl, 2);
}

int launch_dp_allreduce_sgd(const DpState& st, double* params, double* grads, double scale, cudaStream_t stream,
                            long long* cursor, long long batch, long long n_samples, const double* stats, double* stats_ring,
                            bool already_pushed, Timeline* tl) {
    if (!st.connected) return fail(RCN_ERR_STATE, "data-parallel group is not connected");
    if (st.n == 0) return RCN_OK;
    DpPush pp = dp_push_desc(st);
    pp.tl = tl;
    // rcn's canonical network (23 860 parameters): <= 20 fat CTAs, so that kernel A of the next step (128 CTAs, a whole SM
    // each) runs beside this kernel; larger buffers are bandwidth work and spread over the machine
    unsigned grid = cdiv(st.n, kDpThreads);
    if (grid <= 2u * kDpMaxCtas) { if (grid > (unsigned)kDpMaxCtas) grid = kDpMaxCtas; }
    else if (grid > 2u * kNumSMs) grid = 2u * kNumSMs;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(kDpThreads, 1, 1);
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const int pushed_i = already_pushed ? 1 : 0;
#define RCN_DP_LAUNCH(W)                                                                                                       \
    RCN_LAUNCH("dp_allreduce_sgd_kernel", stream,                                                                              \
               cudaLaunchKernelEx(&cfg, dp_allreduce_sgd_kernel<W>, pp, params, grads, scale, cursor, batch, n_samples, stats,  \
                                  stats_ring, pushed_i))
    switch (st.world) {
        case 2: RCN_DP_LAUNCH(2); break;
        case 4: RCN_DP_LAUNCH(4); break;
        case 8: RCN_DP_LAUNCH(8); break;
        default: RCN_DP_LAUNCH(0); break;
    }
#undef RCN_DP_LAUNCH
    return RCN_OK;
}

}  // namespace rcn
