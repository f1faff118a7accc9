// model.cu -- the C ABI of librcn_cuda.so (include/rcn_cuda.h): model handle, device buffers, host<->device
// staging, and the layer dispatch that replaces rcn's per-sample CPU loops (rcn/src/rcn.rs) with batched
// kernels (features.cu, dense.cu).
#include <cuda.h>
#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <tuple>
#include <vector>

#include "cnn.cuh"
#include "dense.cuh"
#include "features.cuh"
#include "smallnet.cuh"
#include "opctx.cuh"
#include "dp.cuh"
#include "ozaki.cuh"

namespace rcn {

std::string& last_error_ref() {
    thread_local std::string s;
    return s;
}

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return code;
}

// ---- launch accounting / per-kernel event timing --------------------------------------------------------
namespace {
struct ProfRecord { const char* name; cudaEvent_t start, stop; };
std::atomic<unsigned long long> g_launches{0};
std::atomic<bool> g_profiling{false};
std::mutex g_prof_mu;
std::vector<ProfRecord> g_prof;
}  // namespace

LaunchScope::LaunchScope(const char* name, cudaStream_t s) : stream(s), slot(-1) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (!g_profiling.load(std::memory_order_relaxed)) return;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) { cudaGetLastError(); return; }
    ProfRecord r{name, nullptr, nullptr};
    if (cudaEventCreate(&r.start) != cudaSuccess || cudaEventCreate(&r.stop) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(r.start, s);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(r);
    slot = (int)g_prof.size() - 1;
}

LaunchScope::~LaunchScope() {
    if (slot < 0) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (slot < (int)g_prof.size()) cudaEventRecord(g_prof[slot].stop, stream);
}

// ---- streaming from a pinned HOST dataset (rcn_cuda_train_epoch_host fast path) ---------------------------------------
// State block in device memory: [0] cursor (samples, advanced by the update), [3] images arrived in the ring so far; the
// other words are padding.  The step's labels follow.
constexpr int kHsStateSlots = 6;
// the streamed epoch's cursor never wraps (every call re-initialises the state block), so the captured graphs are independent
// of the epoch length and serve every later call with the same batch shape
constexpr long long kHsNoWrap = 1ll << 62;
// consecutive steps captured into one CUDA graph by rcn_cuda_train_epoch_host (RCN_CUDA_HOST_STEPS_PER_GRAPH overrides)
// Default 40: the steps inside a graph follow each other without the host or the PCIe link in between, while every graph
// boundary cost 4-5 us (and now and then 27 us) with copies in flight on the link (profiles/r2_e2e_timeline.txt): 24.8 / 23.4 /
// 22.3 / 21.8 us per step at 5 / 10 / 20 / 40.
static int hs_steps_per_graph() {
    static const int v = []() { const char* e = getenv("RCN_CUDA_HOST_STEPS_PER_GRAPH"); int n = e ? atoi(e) : 0; return n < 1 ? 0 : (n > 64 ? 64 : n); }();
    return v ? v : 40;
}
// How the images of the streamed epoch cross PCIe: the copy engine.  The copy stream walks the dataset with back-to-back
// cudaMemcpyAsync calls into a ring of `kHsRingSteps` chunks, an event behind each; a second stream waits for each event and
// publishes, with an 8-byte copy from a pinned table, how many images have landed (state[3]).  Kernel A's image-loading lanes
// wait for their own image on that counter (wait_arrived), so the compute stream carries nothing but back-to-back graph
// launches -- no events, no per-step join.  Once per quarter of the ring the copy stream waits (cuStreamWaitValue64) until the
// training cursor (state[0]) has passed the quarter's previous occupants.  Copies ramp 1 ... 2 ... 4 ... 8 chunks: the first
// step starts after ONE chunk has crossed the link, later copies run at the link's large-transfer rate.  Measured on a warm
// link (profiles/r2_pcie_dma.json): 43.6 GB/s for one 0.8 MB chunk, 48.7 for two, 53.6 for eight, against 38 GB/s for
// SM-issued zero-copy loads; and no CTA of the step's kernels shares its SM with a copy kernel.  (Publishing the counter on
// the copy stream itself -- cuStreamWriteValue64 or the 8-byte copy -- put ~22 us between consecutive data copies, which then
// no longer pipeline: a one-chunk copy took 40 us instead of 18 and the copy stream became the bottleneck.)  Round 1's
// design -- a prefetch kernel pulling each chunk with zero-copy loads on a parallel graph branch -- measured slower end to
// end (42.8-43.9 M against 48.5-49.5 M images/s) and was removed.  The call streams only when the steps on the ring run
// kernel A with the staged front end (fused_front, the rule of every training step) and the device has 64-bit stream
// memory operations; otherwise it takes the general double-buffered loop.
constexpr size_t kHsRingSteps = 64;   // chunks the ring holds
constexpr size_t kHsQuarter = kHsRingSteps / 4;   // granularity of the copy stream's wait for free ring slots
constexpr size_t kHsMaxCopy = 8;      // chunks per cudaMemcpyAsync once the ramp is over (divides kHsQuarter)
constexpr int kHsEvents = 64;         // one event behind each copy, reused round robin
struct StreamMemOps {
    CUresult (*wait64)(CUstream, CUdeviceptr, cuuint64_t, unsigned int) = nullptr;

    bool ok = false;
};
static const StreamMemOps& stream_mem_ops(int device) {
    static const StreamMemOps ops = [device]() {
        StreamMemOps o;
        auto entry = [](const char* name) -> void* {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return nullptr; }
            return p;
        };
        auto get_attr = reinterpret_cast<CUresult (*)(int*, CUdevice_attribute, CUdevice)>(entry("cuDeviceGetAttribute"));
        o.wait64 = reinterpret_cast<decltype(o.wait64)>(entry("cuStreamWaitValue64"));

        int can = 0;
        o.ok = get_attr && o.wait64 && get_attr(&can, CU_DEVICE_ATTRIBUTE_CAN_USE_64_BIT_STREAM_MEM_OPS, device) == CUDA_SUCCESS && can;
        return o;
    }();
    return ops;
}
bool is_pinned_host_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost && a.devicePointer != nullptr;
}

// Grow-only pinned host table of `T`: the host-side counterpart of DevBuf.
template <typename T> struct PinnedBuf {
    T* p = nullptr;
    size_t cap = 0;
    int reserve(size_t n) {
        if (n <= cap) return RCN_OK;
        release();
        RCN_CUDA_TRY(cudaHostAlloc((void**)&p, n * sizeof(T), cudaHostAllocDefault));
        cap = n;
        return RCN_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// What rcn_cuda_train_epoch_host keeps between calls: two streams beside the model's, their events, the device buffers and
// pinned tables of both loops, and the streamed loop's step graphs with the key they were captured under.
struct HostEpoch {
    cudaStream_t copy_stream = nullptr;        // the H2D copies of the images
    cudaStream_t flag_stream = nullptr;        // streamed loop: publishes the arrival counter behind each copy
    cudaEvent_t fork = nullptr;                // orders another stream after the compute stream
    cudaEvent_t ev_copied[2] = {}, ev_consumed[2] = {};   // double-buffered loop: one pair per staging slot
    cudaEvent_t ev_arrived[kHsEvents] = {};    // streamed loop: one behind each copy, reused round robin
    DevBuf host_slot[2];                       // double-buffered loop: the staging slots
    DevBuf ring, state;                        // streamed loop: kHsRingSteps chunks; state block (kHsStateSlots) | step labels
    PinnedBuf<double> stats;                   // {cost, hits} of every step
    PinnedBuf<long long> counts;               // streamed loop: the "images arrived" value behind each copy
    std::map<int, cudaGraphExec_t> graphs;     // streamed loop: g consecutive steps per graph, captured on first use
    struct Key {
        size_t B = 0, H = 0, W = 0;
        unsigned long long alloc_gen = 0;      // no device buffer has moved since the capture (common.cuh)
        uint64_t mean_bits = 0, sd_bits = 0;   // scale_set travels BY VALUE in the captured kernel arguments
        double scale = 0.0;
        const void *labels = nullptr, *stats = nullptr, *ring = nullptr, *state = nullptr, *grads = nullptr;
        cudaStream_t stream = nullptr;
        bool dp = false;
        long long window = 0;                  // ring size in images (captured in kernel A's arguments)
        auto fields() const { return std::tie(B, H, W, alloc_gen, mean_bits, sd_bits, scale, labels, stats, ring, state, grads, stream, dp, window); }
        bool operator==(const Key& o) const { return fields() == o.fields(); }
    } key;

    int setup() {
        for (cudaStream_t* s : {&copy_stream, &flag_stream})
            if (!*s) RCN_CUDA_TRY(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
        for (cudaEvent_t* e : {&fork, &ev_copied[0], &ev_copied[1], &ev_consumed[0], &ev_consumed[1]})
            if (!*e) RCN_CUDA_TRY(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        for (cudaEvent_t& e : ev_arrived)
            if (!e) RCN_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        return RCN_OK;
    }
    void release() {
        if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
        if (flag_stream) cudaStreamDestroy(flag_stream);
        for (cudaEvent_t e : {fork, ev_copied[0], ev_copied[1], ev_consumed[0], ev_consumed[1]})
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : ev_arrived)
            if (e) cudaEventDestroy(e);
        for (auto& kv : graphs) cudaGraphExecDestroy(kv.second);
        for (DevBuf* b : {&host_slot[0], &host_slot[1], &ring, &state}) b->release();
        stats.release();
        counts.release();
        *this = HostEpoch{};
    }
};

}  // namespace rcn

using namespace rcn;

struct rcn_cuda_model {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    size_t classes = 0;
    std::vector<int32_t> cfg;
    std::vector<size_t> ff;

    // parameters: flat [W0|b0|W1|b1|...], W_l column-major rows[l] x cols[l] (serialization.rs:19-22 order)
    bool params_ready = false;
    std::vector<size_t> rows, cols, w_off, b_off;
    size_t n_params = 0, sum_rows = 0;
    DevBuf params, grads_own;
    double* grads = nullptr;
    bool grads_bound = false;
    double mean = 1.0, sd = 1.0;  // scale_set starts at (1, 1)  (rcn.rs:71)
    SmallNetDesc small_desc{};      // fused path for narrow networks (smallnet.cu)
    bool use_small = false;
    int head = RCN_HEAD_SIGMOID_QUADRATIC;   // output layer and cost: only the convolutional network sets another (model_set_head)

    // feature plan cache
    bool plan_valid = false;
    size_t plan_H = 0, plan_W = 0;
    FeaturePlan plan;
    FeatureScratch fscratch;

    // scratch (grow-only)
    DevBuf in_stage, tgt_stage, feats, acts, deltas, gemm_ws, out_stage, small, red_ws;
    ReduceScratch rs;           // deterministic two-stage reductions (bias gradient, batch statistics)
    ReduceScratch eval_rs;      // per-tile partials + ticket of the inference kernel (rcn_cuda_evaluate_images)
    // epoch mode (rcn.rs:144-149 on a resident dataset)
    const void* ep_images = nullptr;
    const int64_t* ep_labels = nullptr;
    const int64_t* ep_perm = nullptr;
    int ep_fmt = 0;
    size_t ep_n = 0, ep_H = 0, ep_W = 0, ep_B = 0;
    DevBuf ep_state;            // kEpSlots int64 state words (features.cuh: the cursor) | labels_batch [B]
    size_t last_B = 0;          // batch of the last accumulate call (taps)
    bool stats_valid = false;
    // data-parallel group (dp.cu) and the pipelined host-dataset loop (rcn_cuda_train_epoch_host)
    DpState dp;
    bool x_owns_cursor = false;     // an exchange kernel that advances a cursor may be in flight: kernel A must not read the
                                    // cursor ahead of its griddepcontrol.wait (cleared wherever the stream is drained)
    bool dp_pushed = false;         // the last accumulate pushed its gradients to the peers itself (kernel B epilogue)
    DevBuf timeline;                // device-side launch timeline (timeline.cuh), allocated by rcn_cuda_timeline_enable
    bool tl_on = false;
    OzakiWorkspace oz;              // tcgen05 integer-slice GEMM scratch (wide dense layers)
    HostEpoch host_epoch;           // rcn_cuda_train_epoch_host

    double* act(size_t l, size_t B) const {
        size_t off = 0;
        for (size_t j = 0; j < l; ++j) off += rows[j];
        return acts.as<double>() + off * B;
    }
    double* delta(size_t l, size_t B) const {
        size_t off = 0;
        for (size_t j = 0; j < l; ++j) off += rows[j];
        return deltas.as<double>() + off * B;
    }
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() { /* leave the device selected: one process drives one GPU */ }
};

#define RCN_ENTER(h)                                                                     \
    if (!(h)) return fail(RCN_ERR_INVALID, "null model handle");                         \
    DeviceGuard _guard((h)->device);                                                     \
    if (!_guard.ok) return fail(RCN_ERR_CUDA, "cudaSetDevice(%d) failed", (h)->device);

// Consumes the "already pushed" flag of the last accumulate: every push is matched by exactly one receive.
bool take_dp_pushed(rcn_cuda_model* h) {
    const bool p = h->dp_pushed;
    h->dp_pushed = false;
    return p;
}

int ensure_plan(rcn_cuda_model* h, size_t H, size_t W) {
    if (h->plan_valid && h->plan_H == H && h->plan_W == W) return RCN_OK;
    if (H == 0 || W == 0 || H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "bad image size %zu x %zu", H, W);
    RCN_TRY(plan_features(h->cfg.data(), h->cfg.size(), H, W, &h->plan));
    h->plan_valid = true; h->plan_H = H; h->plan_W = W;
    return RCN_OK;
}

size_t pixel_bytes(int fmt) { return fmt == RCN_PIXELS_U8_ROWMAJOR ? 1 : 8; }

// Copies a device result to a possibly-host destination; `synced` is set when the stream was drained.
int deliver(rcn_cuda_model* h, void* dst, const void* dev_src, size_t bytes) {
    if (bytes == 0) return RCN_OK;
    if (is_device_ptr(dst)) {
        if (dst != dev_src) RCN_CUDA_TRY(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return RCN_OK;
    }
    RCN_CUDA_TRY(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int require_params(rcn_cuda_model* h) {
    if (!h->params_ready) return fail(RCN_ERR_STATE, "parameters not initialised: call rcn_cuda_init_params first");
    return RCN_OK;
}

// features (+ optional standardise) into h->feats for device or host images
int features_into(rcn_cuda_model* h, const void* images, int fmt, size_t B, size_t H, size_t W, bool standardise,
                  double* out_dev) {
    RCN_TRY(ensure_plan(h, H, W));
    if (fmt != RCN_PIXELS_U8_ROWMAJOR && fmt != RCN_PIXELS_F64_COLMAJOR) return fail(RCN_ERR_INVALID, "unknown pixel format %d", fmt);
    if (B == 0 || h->plan.L == 0) return RCN_OK;
    if (!images) return fail(RCN_ERR_INVALID, "null images");
    StagedIn in;
    RCN_TRY(in.stage(images, B * H * W * pixel_bytes(fmt), h->in_stage, h->stream, nullptr));
    return launch_features(h->plan, in.dev, fmt, B, H, W, standardise, h->mean, h->sd, out_dev, h->fscratch, h->stream);
}

// forward pass over device feats (cols[0] x B); fills acts; last layer also fills deltas when targets given.  With the
// softmax head the last layer's activations are the logits z instead, and its deltas are left to the head kernel.
int forward_dev(rcn_cuda_model* h, const double* feats, size_t B, const double* onehot, const int64_t* labels,
                bool want_delta) {
    const size_t n = h->rows.size();
    RCN_TRY(h->acts.reserve(h->sum_rows * B * sizeof(double)));
    if (want_delta) RCN_TRY(h->deltas.reserve(h->sum_rows * B * sizeof(double)));
    if (h->use_small && !want_delta)
        return launch_smallnet_forward(h->small_desc, h->params.as<double>(), const_cast<double*>(feats), B,
                                       h->acts.as<double>(), nullptr, h->stream);
    for (size_t l = 0; l < n; ++l) {
        const double* a_in = l == 0 ? feats : h->act(l - 1, B);
        const bool last = (l + 1 == n);
        if (last && h->head == RCN_HEAD_SOFTMAX_XENT) {   // logits; the head kernel computes p and the output delta
            RCN_TRY(launch_dense_logits(h->params.as<double>() + h->w_off[l], h->params.as<double>() + h->b_off[l], a_in, h->rows[l],
                                        h->cols[l], B, h->act(l, B), h->stream, &h->oz));
            break;
        }
        RCN_TRY(launch_dense_forward(h->params.as<double>() + h->w_off[l], h->params.as<double>() + h->b_off[l], a_in,
                                     h->rows[l], h->cols[l], B, h->act(l, B),
                                     (last && want_delta) ? h->delta(l, B) : nullptr, onehot, labels, h->stream, &h->oz));
    }
    return RCN_OK;
}

// What a training step asks of the accumulate.  On the fused small-network path kernel B applies `upd` itself: on one GPU
// the whole update, on a data-parallel group (`upd.params` null) only the cursor / result ring, and the exchange kernel
// updates.  `push`: on a connected group kernel B pushes its gradients to the peers -- not in a warm-up, as every push is
// consumed by exactly one receive.  The default request arms nothing.
struct StepRequest {
    SnUpdate upd{};
    bool push = true;
};

// What kernel B did with the request's update; finish_step launches the rest.
enum class StepDone {
    nothing,   // the generic path, an over-size batch, or no update armed
    cursor,    // advanced the cursor and wrote the result ring (data-parallel group)
    update,    // updated the parameters (one GPU): the step is complete
};

// The update of a training step: `scale` = eta / global batch; the optional device-side cursor advances by `batch` over
// `n_samples`, and `stats_ring` receives each step's {cost, hits}.  `streamed`: kernel A of the streamed host epoch reads
// the cursor ahead of its wait (one GPU).
SnUpdate step_update(rcn_cuda_model* h, double scale, long long* cursor = nullptr, long long batch = 0, long long n_samples = 0,
                     double* stats_ring = nullptr, bool streamed = false) {
    SnUpdate u{};
    // (Receiving inside kernel B on a group as well was measured slower, 2 GPUs, c2: 30.8 vs 28.4 us/step -- the NVLink
    // round trip is then exposed inside the kernel instead of overlapping the next launch -- and was removed.)
    if (!h->dp.connected) u.params = h->params.as<double>();
    u.scale = scale;
    u.cursor = cursor;
    u.batch = batch;
    u.n_samples = n_samples;
    u.stats_ring = stats_ring;
    u.early_cursor = (!h->dp.connected && streamed) ? 1 : 0;
    return u;
}

// Launches what kernel B left of a step: on a data-parallel group the exchange kernel (receive, sum, update), otherwise the
// update kernel; either advances the cursor and writes the result ring unless kernel B already did.
int finish_step(rcn_cuda_model* h, const SnUpdate& u, StepDone done) {
    if (done == StepDone::update) return RCN_OK;
    long long* cursor = done == StepDone::cursor ? nullptr : u.cursor;
    const double* stats = u.stats_ring ? h->small.as<double>() : nullptr;   // the step's {cost, hits}, written by the accumulate
    if (h->dp.connected) {
        if (cursor) h->x_owns_cursor = true;
        return launch_dp_allreduce_sgd(h->dp, h->params.as<double>(), h->grads, u.scale, h->stream, cursor, u.batch, u.n_samples,
                                       stats, u.stats_ring, take_dp_pushed(h), h->small_desc.tl);
    }
    return launch_sgd_update(h->params.as<double>(), h->grads, h->n_params, u.scale, h->stream, cursor, u.batch, u.n_samples, stats,
                             u.stats_ring);
}

int accumulate_dev(rcn_cuda_model* h, const double* feats, const double* onehot, const int64_t* labels, size_t B,
                   const SmallNetFront* front, const StepRequest& req, StepDone* done) {
    const size_t n = h->rows.size();
    if (done) *done = StepDone::nothing;
    if (h->dp_pushed)   // a pushed gradient must be received by the group's update before the next one is produced
        return fail(RCN_ERR_STATE, "data-parallel group: the previous gradients were pushed to the peers but never applied "
                                   "(every accumulate needs exactly one apply on every rank)");
    if (B == 0) {
        RCN_CUDA_TRY(cudaMemsetAsync(h->grads, 0, h->n_params * sizeof(double), h->stream));
        return RCN_OK;
    }
    if (h->use_small && B <= smallnet_max_batch()) {
        RCN_TRY(h->acts.reserve(h->sum_rows * B * sizeof(double)));
        RCN_TRY(h->deltas.reserve(h->sum_rows * B * sizeof(double)));
        RCN_TRY(h->small.reserve(64));
        DpPush push{};
        const bool fuse_push = h->dp.connected && req.push;
        if (fuse_push) push = dp_push_desc(h->dp);
        const SnUpdate& upd = req.upd;
        const bool armed = (upd.params || upd.cursor) && (!h->dp.connected || fuse_push);
        RCN_TRY(launch_smallnet_backprop(h->small_desc, h->params.as<double>(), const_cast<double*>(feats), B, onehot,
                                         labels, h->acts.as<double>(), h->deltas.as<double>(), h->grads,
                                         h->small.as<double>(), h->gemm_ws, front, h->stream, fuse_push ? &push : nullptr,
                                         armed ? &upd : nullptr));
        if (done) *done = upd.params ? StepDone::update : (armed && upd.cursor) ? StepDone::cursor : StepDone::nothing;
        h->dp_pushed = fuse_push;   // pushed but not yet received: the exchange kernel must follow
        h->stats_valid = true;
        h->last_B = B;
        return RCN_OK;
    }
    if (front) return fail(RCN_ERR_STATE, "internal: fused front end requested on the generic path");
    const bool softmax = h->head == RCN_HEAD_SOFTMAX_XENT;
    if (softmax && !labels) return fail(RCN_ERR_INVALID, "the softmax head takes labels, not one-hot targets");
    RCN_TRY(forward_dev(h, feats, B, onehot, labels, true));
    RCN_TRY(h->small.reserve(64));
    if (softmax)   // p over z, delta_L = p - onehot(label), and the batch {cost, hits}
        RCN_TRY(launch_softmax_xent_head(h->act(n - 1, B), h->rows[n - 1], B, labels, h->delta(n - 1, B), nullptr,
                                         h->small.as<double>(), h->rs, h->stream));
    for (size_t l = n - 1; l-- > 0;)  // rcn.rs:305-311
        RCN_TRY(launch_dense_backward_data(h->params.as<double>() + h->w_off[l + 1], h->delta(l + 1, B), h->act(l, B),
                                           h->rows[l], h->rows[l + 1], B, h->delta(l, B), h->stream, &h->oz));
    for (size_t l = 0; l < n; ++l) {
        const double* a_prev = l == 0 ? feats : h->act(l - 1, B);
        RCN_TRY(launch_dense_backward_weight(h->delta(l, B), a_prev, h->rows[l], h->cols[l], B, h->grads + h->w_off[l],
                                             h->grads + h->b_off[l], h->gemm_ws, h->rs, h->stream, &h->oz));
    }
    if (!softmax)
        RCN_TRY(launch_batch_stats(h->act(n - 1, B), h->rows[n - 1], B, onehot, labels, h->small.as<double>(), h->rs, h->stream));
    h->stats_valid = true;
    h->last_B = B;
    return RCN_OK;
}

// Does kernel A run the convpool stack of these DEVICE images itself?  It does for a narrow network, u8 pixels and a stack
// it implements, when the front end selected for these images (the staged one where it qualifies, else the generic one)
// fits its shared memory.  Fills `fr` with that front end, standardised with scale_set; `bi` optional, see below.
bool fused_front(const rcn_cuda_model* h, const void* images, int fmt, size_t H, size_t W, const BatchIndex* bi,
                 SmallNetFront* fr) {
    if (!h->use_small || fmt != RCN_PIXELS_U8_ROWMAJOR || h->plan.n_conv > 10 || h->plan.L == 0) return false;
    *fr = SmallNetFront{};
    fr->images = (const uint8_t*)images;
    fr->H = (int)H; fr->W = (int)W;
    fr->max_elems = (int)h->plan.max_elems;
    fr->stages = h->plan.stages;
    fr->sc = make_standardise(h->plan, RCN_PIXELS_U8_ROWMAJOR, true, h->mean, h->sd);
    if (bi) fr->bi = *bi;
    smallnet_front_select(h->plan, fr);
    return smallnet_front_fits(h->small_desc, *fr);
}

// images (DEVICE) -> gradient sums.  The canonical narrow network with u8 pixels runs the convpool stack inside
// kernel A (smallnet.cu); everything else runs the feature kernel(s) first.  `bi` (optional) is the epoch-mode
// device-side batch selection; without it `labels` are this batch's labels.
int accumulate_images_dev(rcn_cuda_model* h, const void* images, int fmt, const int64_t* labels, size_t B, size_t H,
                          size_t W, const BatchIndex* bi, const StepRequest& req = {}, StepDone* done = nullptr) {
    RCN_TRY(h->feats.reserve(h->plan.L * B * sizeof(double)));
    const int64_t* step_labels = bi ? (const int64_t*)bi->labels_batch : labels;
    SmallNetFront fr;
    if (B <= smallnet_max_batch() && fused_front(h, images, fmt, H, W, bi, &fr)) {
        // Data-parallel step behind the exchange kernel: kernel A may run its front end ahead of griddepcontrol.wait
        // (smallnet.cu) when this step's kernel B pushes to the peers (so the exchange kernel X precedes the next kernel
        // A) and any device-side cursor it reads is advanced by kernel B -- this step's and the previous one's
        // (x_owns_cursor) -- not by X, which may still be running then.
        fr.prewait = (fr.use_cp && h->dp.connected && req.push && !h->x_owns_cursor &&
                      (!fr.bi.cursor || req.upd.cursor == fr.bi.cursor)) ? 1 : 0;
        // One GPU, streamed host epoch: the same front end under the tail of the previous step's kernel B (which triggers its
        // dependents early).  Safe whatever precedes this launch: a kernel that does not trigger early has completed before
        // kernel A starts; kernel B advances a device-side cursor before it triggers, and the only buffer both touch -- the
        // features -- is written by this kernel A after its wait.  Measured: the host epoch gains 3-6 % (the arrival-counter
        // wait and the ring loads move under kernel B).  Prewaiting nowhere, or in every training step, measured slower and
        // was removed: in the device-resident step kernel A needs a whole SM's registers, so all but ~26 of its CTAs start
        // only when kernel B's CTAs leave, and its parameter loads are no longer hidden behind the front end.
        if (!h->dp.connected && fr.use_cp && fr.bi.window != 0) fr.prewait = 2;
        return accumulate_dev(h, h->feats.as<double>(), nullptr, step_labels, B, &fr, req, done);
    }
    RCN_TRY(launch_features(h->plan, images, fmt, B, H, W, true, h->mean, h->sd, h->feats.as<double>(), h->fscratch,
                            h->stream, bi));
    return accumulate_dev(h, h->feats.as<double>(), nullptr, step_labels, B, nullptr, req, done);
}

// stage targets (exactly one of onehot / labels)
int stage_targets(rcn_cuda_model* h, const double* onehot, const int64_t* labels, size_t B, const double** oh_dev,
                  const int64_t** lb_dev) {
    *oh_dev = nullptr; *lb_dev = nullptr;
    if ((onehot == nullptr) == (labels == nullptr))
        return fail(RCN_ERR_INVALID, "exactly one of onehot / labels must be given");
    StagedIn in;
    if (onehot) {
        RCN_TRY(in.stage(onehot, h->classes * B * sizeof(double), h->tgt_stage, h->stream, nullptr));
        *oh_dev = (const double*)in.dev;
    } else {
        RCN_TRY(in.stage(labels, B * sizeof(int64_t), h->tgt_stage, h->stream, nullptr));
        *lb_dev = (const int64_t*)in.dev;
    }
    return RCN_OK;
}

int check_feature_width(rcn_cuda_model* h, size_t L) {
    if (h->cols[0] != L)  // nalgebra `w * a` dimension mismatch (reference panics; see rcn.rs:443 quirk)
        return fail(RCN_ERR_SHAPE, "Matrix multiplication dimensions mismatch: first layer expects %zu inputs, feature vector has %zu",
                    h->cols[0], L);
    return RCN_OK;
}

}  // namespace

extern "C" {

const char* rcn_cuda_last_error(void) { return last_error_ref().c_str(); }
int rcn_cuda_version(void) { return 100; }

int rcn_cuda_device_count(int* count) {
    if (!count) return fail(RCN_ERR_INVALID, "null count");
    RCN_CUDA_TRY(cudaGetDeviceCount(count));
    return RCN_OK;
}

int rcn_cuda_create(size_t classes, const int32_t* convpool_cfg, size_t n_convpool, const size_t* feedforward_cfg,
                    size_t n_feedforward, int device, rcn_cuda_handle* out) {
    if (!out) return fail(RCN_ERR_INVALID, "null out handle");
    *out = nullptr;
    if (n_convpool && !convpool_cfg) return fail(RCN_ERR_INVALID, "null convpool_cfg");
    if (n_feedforward && !feedforward_cfg) return fail(RCN_ERR_INVALID, "null feedforward_cfg");
    for (size_t i = 0; i < n_convpool; ++i)
        if (convpool_cfg[i] < 0 || convpool_cfg[i] > 3) return fail(RCN_ERR_INVALID, "unknown RCNLayer code %d", convpool_cfg[i]);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(RCN_ERR_CUDA, "no CUDA device available (%s); librcn_cuda has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= ndev) return fail(RCN_ERR_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
    RCN_CUDA_TRY(cudaSetDevice(device));
    std::unique_ptr<rcn_cuda_model> m(new (std::nothrow) rcn_cuda_model());
    if (!m) return fail(RCN_ERR_INVALID, "out of host memory");
    m->device = device;
    m->classes = classes;
    m->cfg.assign(convpool_cfg, convpool_cfg + n_convpool);
    m->ff.assign(feedforward_cfg, feedforward_cfg + n_feedforward);
    RCN_CUDA_TRY(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
    m->stream = m->own_stream;
    *out = m.release();
    return RCN_OK;
}

int rcn_cuda_destroy(rcn_cuda_handle h) {
    if (!h) return RCN_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->own_stream) { cudaStreamSynchronize(h->own_stream); cudaStreamDestroy(h->own_stream); }
    h->host_epoch.release();
    dp_release(h->dp);
    h->oz.release();
    DevBuf* bufs[] = {&h->params, &h->grads_own, &h->in_stage, &h->tgt_stage, &h->feats, &h->acts, &h->deltas,
                      &h->gemm_ws, &h->out_stage, &h->small, &h->red_ws, &h->ep_state, &h->fscratch.a, &h->fscratch.b, &h->rs.buf,
                      &h->eval_rs.buf};
    for (DevBuf* b : bufs) b->release();
    delete h;
    return RCN_OK;
}

int rcn_cuda_set_stream(rcn_cuda_handle h, void* cuda_stream) {
    RCN_ENTER(h);
    h->stream = (cuda_stream == RCN_STREAM_OWN) ? h->own_stream : (cudaStream_t)cuda_stream;
    return RCN_OK;
}

static void stream_drained(rcn_cuda_model* h);

int rcn_cuda_synchronize(rcn_cuda_handle h) {
    RCN_ENTER(h);
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    return RCN_OK;
}

int rcn_cuda_feature_shape(rcn_cuda_handle h, size_t H, size_t W, size_t* n_maps, size_t* map_h, size_t* map_w) {
    RCN_ENTER(h);
    RCN_TRY(ensure_plan(h, H, W));
    if (n_maps) *n_maps = h->plan.n_maps;
    if (map_h) *map_h = h->plan.map_h;
    if (map_w) *map_w = h->plan.map_w;
    return RCN_OK;
}

namespace {
// Installs explicit layer shapes (rows[i] x cols[i]), allocates zeroed parameters / gradients, picks the fused path.
int install_shapes(rcn_cuda_model* h, const std::vector<size_t>& rows, const std::vector<size_t>& cols) {
    const size_t n = rows.size();
    // a captured step holds the layer shapes by value (SmallNetDesc): new shapes invalidate it like a moved buffer does
    alloc_generation().fetch_add(1, std::memory_order_relaxed);
    h->rows.clear(); h->cols.clear(); h->w_off.clear(); h->b_off.clear();
    size_t off = 0, sum_rows = 0;
    for (size_t i = 0; i < n; ++i) {
        if (rows[i] == 0) return fail(RCN_ERR_INVALID, "layer %zu has zero neurons", i);
        h->rows.push_back(rows[i]); h->cols.push_back(cols[i]);  // dims = (output_size, input_size)  (rcn.rs:502)
        h->w_off.push_back(off); off += rows[i] * cols[i];
        h->b_off.push_back(off); off += rows[i];
        sum_rows += rows[i];
    }
    h->n_params = off; h->sum_rows = sum_rows;
    {   // fused small-network path (smallnet.cu) unless RCN_CUDA_SMALLNET=0
        SmallNetDesc d{};
        h->use_small = false;
        const char* env = getenv("RCN_CUDA_SMALLNET");
        if (n <= (size_t)kSmallNetMaxLayers && h->cols[0] >= 1 && h->cols[0] < (1u << 24) && off < (1u << 30) &&
            !(env && env[0] == '0')) {
            d.n_layers = (int)n; d.n_in = (int)h->cols[0]; d.n_params = (int)off;
            for (size_t i = 0; i < n; ++i) { d.rows[i] = (int)h->rows[i]; d.w_off[i] = (int)h->w_off[i]; d.b_off[i] = (int)h->b_off[i]; }
            bool ok = true;
            for (size_t i = 0; i < n; ++i) ok = ok && h->rows[i] <= 32;
            ok = ok && h->head == RCN_HEAD_SIGMOID_QUADRATIC;   // kernels A/B implement the sigmoid / quadratic head only
            if (ok && smallnet_eligible(d)) { h->small_desc = d; h->small_desc.tl = h->tl_on ? h->timeline.as<Timeline>() : nullptr; h->use_small = true; }
        }
    }
    RCN_TRY(h->params.reserve(off * sizeof(double)));
    RCN_CUDA_TRY(cudaMemsetAsync(h->params.p, 0, off * sizeof(double), h->stream));
    if (!h->grads_bound) {
        RCN_TRY(h->grads_own.reserve(off * sizeof(double)));
        h->grads = h->grads_own.as<double>();
        RCN_CUDA_TRY(cudaMemsetAsync(h->grads, 0, off * sizeof(double), h->stream));
    }
    h->params_ready = true;
    h->stats_valid = false;
    return RCN_OK;
}
}  // namespace

int rcn_cuda_init_params(rcn_cuda_handle h, size_t l) {
    RCN_ENTER(h);
    // load_weights_and_bias (rcn.rs:425-457)
    if (h->ff.empty()) return fail(RCN_ERR_OUT_OF_BOUNDS, "index out of bounds: feedforward_cfg is empty (rcn.rs:444)");
    unsigned c = 0, p = 0;
    for (int32_t layer : h->cfg) {
        if (layer == RCN_LAYER_CONV_NONE || layer == RCN_LAYER_CONV_SAME) c += 1; else p += 2;
    }
    if (c > 20 || p > 60) return fail(RCN_ERR_INVALID, "convpool stack too deep");
    size_t pc = 1, pp = 1;
    for (unsigned i = 0; i < c; ++i) pc *= 4;
    for (unsigned i = 0; i < p; ++i) pp *= 2;
    size_t a = pc / pp * l;  // 4^c / 2^p * l, integer division first (rcn.rs:443)
    size_t b = h->ff[0];
    const size_t n = h->ff.size() + 1;
    std::vector<size_t> rows, cols;
    for (size_t i = 0; i < n; ++i) {
        rows.push_back(b); cols.push_back(a);
        a = b;
        b = (i + 1 < h->ff.size()) ? h->ff[i + 1] : h->classes;
    }
    return install_shapes(h, rows, cols);
}

// A deserialized model carries whatever matrices its checkpoint holds (main.rs:50): install explicit shapes.
int rcn_cuda_init_params_shapes(rcn_cuda_handle h, const size_t* rows, const size_t* cols, size_t n_layers) {
    RCN_ENTER(h);
    if (!rows || !cols || n_layers == 0) return fail(RCN_ERR_INVALID, "need at least one layer shape");
    for (size_t i = 1; i < n_layers; ++i)
        if (cols[i] != rows[i - 1])
            return fail(RCN_ERR_SHAPE, "Matrix multiplication dimensions mismatch: layer %zu has %zu inputs, layer %zu has %zu outputs", i,
                        cols[i], i - 1, rows[i - 1]);
    return install_shapes(h, std::vector<size_t>(rows, rows + n_layers), std::vector<size_t>(cols, cols + n_layers));
}

int rcn_cuda_num_layers(rcn_cuda_handle h, size_t* n_layers) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n_layers) *n_layers = h->rows.size();
    return RCN_OK;
}

int rcn_cuda_layer_shape(rcn_cuda_handle h, size_t layer, size_t* rows, size_t* cols) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size()) return fail(RCN_ERR_INVALID, "layer %zu out of range", layer);
    if (rows) *rows = h->rows[layer];
    if (cols) *cols = h->cols[layer];
    return RCN_OK;
}

int rcn_cuda_param_count(rcn_cuda_handle h, size_t* n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n) *n = h->n_params;
    return RCN_OK;
}

static int copy_in(rcn_cuda_handle h, double* dst_dev, const double* src, size_t n) {
    if (!src) return fail(RCN_ERR_INVALID, "null source");
    if (n == 0) return RCN_OK;
    const bool dev = is_device_ptr(src);
    RCN_CUDA_TRY(cudaMemcpyAsync(dst_dev, src, n * sizeof(double), dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
    if (!dev) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));  // pageable source may be reused by the caller
    return RCN_OK;
}

int rcn_cuda_set_weights(rcn_cuda_handle h, size_t layer, size_t rows, size_t cols, const double* w) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size()) return fail(RCN_ERR_INVALID, "layer %zu out of range", layer);
    if (rows != h->rows[layer] || cols != h->cols[layer])
        return fail(RCN_ERR_SHAPE, "weights for layer %zu must be %zu x %zu, got %zu x %zu", layer, h->rows[layer], h->cols[layer], rows, cols);
    return copy_in(h, h->params.as<double>() + h->w_off[layer], w, rows * cols);
}

int rcn_cuda_get_weights(rcn_cuda_handle h, size_t layer, double* w) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size() || !w) return fail(RCN_ERR_INVALID, "bad layer / null destination");
    return deliver(h, w, h->params.as<double>() + h->w_off[layer], h->rows[layer] * h->cols[layer] * sizeof(double));
}

int rcn_cuda_set_bias(rcn_cuda_handle h, size_t layer, size_t n, const double* b) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size()) return fail(RCN_ERR_INVALID, "layer %zu out of range", layer);
    if (n != h->rows[layer]) return fail(RCN_ERR_SHAPE, "bias for layer %zu must have %zu entries, got %zu", layer, h->rows[layer], n);
    return copy_in(h, h->params.as<double>() + h->b_off[layer], b, n);
}

int rcn_cuda_get_bias(rcn_cuda_handle h, size_t layer, double* b) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size() || !b) return fail(RCN_ERR_INVALID, "bad layer / null destination");
    return deliver(h, b, h->params.as<double>() + h->b_off[layer], h->rows[layer] * sizeof(double));
}

int rcn_cuda_set_params(rcn_cuda_handle h, const double* flat, size_t n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n != h->n_params) return fail(RCN_ERR_SHAPE, "model has %zu parameters, got %zu", h->n_params, n);
    return copy_in(h, h->params.as<double>(), flat, n);
}

int rcn_cuda_get_params(rcn_cuda_handle h, double* flat, size_t n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n != h->n_params || !flat) return fail(RCN_ERR_SHAPE, "model has %zu parameters, got %zu", h->n_params, n);
    return deliver(h, flat, h->params.p, n * sizeof(double));
}

int rcn_cuda_set_scale(rcn_cuda_handle h, double mean, double sd) {
    RCN_ENTER(h);
    h->mean = mean; h->sd = sd;
    return RCN_OK;
}

int rcn_cuda_get_scale(rcn_cuda_handle h, double* mean, double* sd) {
    RCN_ENTER(h);
    if (mean) *mean = h->mean;
    if (sd) *sd = h->sd;
    return RCN_OK;
}

int rcn_cuda_features(rcn_cuda_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                      int standardise, double* out) {
    RCN_ENTER(h);
    RCN_TRY(ensure_plan(h, H, W));
    const size_t bytes = h->plan.L * B * sizeof(double);
    if (bytes == 0) return RCN_OK;
    if (!out) return fail(RCN_ERR_INVALID, "null output");
    double* out_dev = out;
    const bool out_is_dev = is_device_ptr(out);
    if (!out_is_dev) { RCN_TRY(h->feats.reserve(bytes)); out_dev = h->feats.as<double>(); }
    RCN_TRY(features_into(h, images, pixel_format, B, H, W, standardise != 0, out_dev));
    if (!out_is_dev) RCN_TRY(deliver(h, out, out_dev, bytes));
    return RCN_OK;
}

int rcn_cuda_gen_scales(rcn_cuda_handle h, const double* feats, size_t L, size_t B, double* mean, double* sd) {
    RCN_ENTER(h);
    if (!feats || L * B == 0) return fail(RCN_ERR_INVALID, "gen_scales needs a non-empty set");
    StagedIn in;
    RCN_TRY(in.stage(feats, L * B * sizeof(double), h->in_stage, h->stream, nullptr));
    RCN_TRY(h->small.reserve(64));
    double* res = h->small.as<double>() + 4;
    RCN_TRY(launch_gen_scales((const double*)in.dev, L * B, res, h->red_ws, h->stream));
    double host[2];
    RCN_CUDA_TRY(cudaMemcpyAsync(host, res, sizeof(host), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    h->mean = host[0]; h->sd = host[1];  // self.scale_set = (mean, sd)  (rcn.rs:249-250)
    if (mean) *mean = host[0];
    if (sd) *sd = host[1];
    return RCN_OK;
}

int rcn_cuda_standardise(rcn_cuda_handle h, double* feats, size_t n) {
    RCN_ENTER(h);
    if (n == 0) return RCN_OK;
    if (!feats) return fail(RCN_ERR_INVALID, "null feats");
    if (is_device_ptr(feats)) return launch_standardise(feats, n, h->mean, h->sd, h->stream);
    RCN_TRY(h->in_stage.reserve(n * sizeof(double)));
    RCN_CUDA_TRY(cudaMemcpyAsync(h->in_stage.p, feats, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    RCN_TRY(launch_standardise(h->in_stage.as<double>(), n, h->mean, h->sd, h->stream));
    return deliver(h, feats, h->in_stage.p, n * sizeof(double));
}

int rcn_cuda_forward(rcn_cuda_handle h, const double* feats, size_t B, double* out_acts) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (B == 0) return RCN_OK;
    if (!feats || !out_acts) return fail(RCN_ERR_INVALID, "null feats / output");
    StagedIn in;
    RCN_TRY(in.stage(feats, h->cols[0] * B * sizeof(double), h->in_stage, h->stream, nullptr));
    RCN_TRY(forward_dev(h, (const double*)in.dev, B, nullptr, nullptr, false));
    const size_t n = h->rows.size();
    return deliver(h, out_acts, h->act(n - 1, B), h->rows[n - 1] * B * sizeof(double));
}

static int classify_dev_feats(rcn_cuda_handle h, const double* feats_dev, size_t B, int64_t* labels_out) {
    RCN_TRY(forward_dev(h, feats_dev, B, nullptr, nullptr, false));
    const size_t n = h->rows.size();
    int64_t* lab_dev = labels_out;
    const bool out_dev = is_device_ptr(labels_out);
    if (!out_dev) { RCN_TRY(h->out_stage.reserve(B * sizeof(int64_t))); lab_dev = h->out_stage.as<int64_t>(); }
    RCN_TRY(launch_argmax_last(h->act(n - 1, B), h->rows[n - 1], B, lab_dev, h->stream));
    if (!out_dev) RCN_TRY(deliver(h, labels_out, lab_dev, B * sizeof(int64_t)));
    return RCN_OK;
}

int rcn_cuda_classify_features(rcn_cuda_handle h, const double* feats, size_t B, int64_t* labels_out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (B == 0) return RCN_OK;
    if (!feats || !labels_out) return fail(RCN_ERR_INVALID, "null feats / output");
    StagedIn in;
    RCN_TRY(in.stage(feats, h->cols[0] * B * sizeof(double), h->in_stage, h->stream, nullptr));
    return classify_dev_feats(h, (const double*)in.dev, B, labels_out);
}

int rcn_cuda_classify(rcn_cuda_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                      int64_t* labels_out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (B == 0) return RCN_OK;
    if (!labels_out) return fail(RCN_ERR_INVALID, "null output");
    RCN_TRY(ensure_plan(h, H, W));
    RCN_TRY(check_feature_width(h, h->plan.L));
    RCN_TRY(h->feats.reserve(h->plan.L * B * sizeof(double)));
    RCN_TRY(features_into(h, images, pixel_format, B, H, W, true, h->feats.as<double>()));  // rcn.rs:84-89
    return classify_dev_feats(h, h->feats.as<double>(), B, labels_out);
}

int rcn_cuda_evaluate(rcn_cuda_handle h, const double* feats, const int64_t* labels, size_t B, uint64_t* accept) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!accept) return fail(RCN_ERR_INVALID, "null accept");
    *accept = 0;
    if (B == 0) return RCN_OK;
    if (!feats || !labels) return fail(RCN_ERR_INVALID, "null feats / labels");
    StagedIn in, lb;
    RCN_TRY(in.stage(feats, h->cols[0] * B * sizeof(double), h->in_stage, h->stream, nullptr));
    RCN_TRY(lb.stage(labels, B * sizeof(int64_t), h->tgt_stage, h->stream, nullptr));
    RCN_TRY(forward_dev(h, (const double*)in.dev, B, nullptr, nullptr, false));
    const size_t n = h->rows.size();
    RCN_TRY(h->small.reserve(64));
    double* st = h->small.as<double>() + 2;
    RCN_TRY(launch_batch_stats(h->act(n - 1, B), h->rows[n - 1], B, nullptr, (const int64_t*)lb.dev, st, h->rs, h->stream));
    uint64_t host[2];
    RCN_CUDA_TRY(cudaMemcpyAsync(host, st, sizeof(host), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    *accept = host[1];
    return RCN_OK;
}

int rcn_cuda_evaluate_images(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B, size_t H,
                             size_t W, double* cost_out, uint64_t* accept_out, int64_t* labels_out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (pixel_format != RCN_PIXELS_U8_ROWMAJOR && pixel_format != RCN_PIXELS_F64_COLMAJOR)
        return fail(RCN_ERR_INVALID, "unknown pixel format %d", pixel_format);
    if (B == 0) {
        if (cost_out && is_device_ptr(cost_out)) RCN_CUDA_TRY(cudaMemsetAsync(cost_out, 0, sizeof(double), h->stream));
        else if (cost_out) *cost_out = 0.0;
        if (accept_out && is_device_ptr(accept_out)) RCN_CUDA_TRY(cudaMemsetAsync(accept_out, 0, sizeof(uint64_t), h->stream));
        else if (accept_out) *accept_out = 0;
        return RCN_OK;
    }
    if (!images || !labels || !cost_out || !accept_out) return fail(RCN_ERR_INVALID, "null images / labels / cost / accept");
    RCN_TRY(ensure_plan(h, H, W));
    RCN_TRY(check_feature_width(h, h->plan.L));
    bool host_in = false;
    StagedIn in, lb;
    RCN_TRY(in.stage(images, B * H * W * pixel_bytes(pixel_format), h->in_stage, h->stream, &host_in));
    RCN_TRY(lb.stage(labels, B * sizeof(int64_t), h->tgt_stage, h->stream, &host_in));
    const int64_t* lab_in = (const int64_t*)lb.dev;
    RCN_TRY(h->small.reserve(64));
    double* st = h->small.as<double>() + 6;   // {cost, hits}: not the words behind rcn_cuda_last_batch_stats (0, 1)
    int64_t* lab_dev = labels_out;
    const bool lab_host = labels_out && !is_device_ptr(labels_out);
    if (lab_host) { RCN_TRY(h->out_stage.reserve(B * sizeof(int64_t))); lab_dev = h->out_stage.as<int64_t>(); }
    SmallNetFront fr;
    if (fused_front(h, in.dev, pixel_format, H, W, nullptr, &fr)) {
        // One launch, the front end inside the inference kernel.  Measured against the feature kernel followed by the
        // inference kernel on the features (profiles/eval_routes_b200.txt, B200 at 1000 W) it was faster from 64 to
        // 1 048 576 images (9.42 against 9.69 ms at 1 048 576) and equal at 1, so that route was not kept.
        RCN_TRY(launch_smallnet_infer(h->small_desc, h->params.as<double>(), B, lab_in, lab_dev, st, h->eval_rs, fr, h->stream));
    } else {   // the existing kernels: features + standardise, forward, batch statistics, argmax
        RCN_TRY(h->feats.reserve(h->plan.L * B * sizeof(double)));
        RCN_TRY(launch_features(h->plan, in.dev, pixel_format, B, H, W, true, h->mean, h->sd, h->feats.as<double>(), h->fscratch,
                                h->stream));
        RCN_TRY(forward_dev(h, h->feats.as<double>(), B, nullptr, nullptr, false));
        const size_t n = h->rows.size();
        RCN_TRY(launch_batch_stats(h->act(n - 1, B), h->rows[n - 1], B, nullptr, lab_in, st, h->rs, h->stream));
        if (labels_out) RCN_TRY(launch_argmax_last(h->act(n - 1, B), h->rows[n - 1], B, lab_dev, h->stream));
    }
    if (lab_host) RCN_TRY(deliver(h, labels_out, lab_dev, B * sizeof(int64_t)));
    RCN_TRY(deliver(h, cost_out, st, sizeof(double)));
    RCN_TRY(deliver(h, accept_out, st + 1, sizeof(uint64_t)));
    if (host_in) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));   // the caller may reuse its host buffers
    return RCN_OK;
}

// The accumulate entry points behind the public ones, which pass the default (unarmed) request; the training steps arm
// their update.
static int accumulate_gradients(rcn_cuda_model* h, const double* feats, const double* onehot, const int64_t* labels, size_t B,
                                const StepRequest& req, StepDone* done) {
    RCN_TRY(require_params(h));
    const double* oh = nullptr; const int64_t* lb = nullptr;
    const double* f_dev = nullptr;
    bool host_in = false;
    if (B) {
        if (!feats) return fail(RCN_ERR_INVALID, "null feats");
        RCN_TRY(stage_targets(h, onehot, labels, B, &oh, &lb));
        StagedIn in;
        RCN_TRY(in.stage(feats, h->cols[0] * B * sizeof(double), h->in_stage, h->stream, &host_in));
        f_dev = (const double*)in.dev;
    }
    RCN_TRY(accumulate_dev(h, f_dev, oh, lb, B, nullptr, req, done));
    if (host_in || (onehot && !is_device_ptr(onehot)) || (labels && !is_device_ptr(labels)))
        RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));  // caller may reuse host buffers
    return RCN_OK;
}

static int accumulate_gradients_images(rcn_cuda_model* h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                                       size_t H, size_t W, const StepRequest& req, StepDone* done) {
    RCN_TRY(require_params(h));
    RCN_TRY(ensure_plan(h, H, W));
    RCN_TRY(check_feature_width(h, h->plan.L));
    const double* oh = nullptr; const int64_t* lb = nullptr;
    if (B) {
        if (!labels) return fail(RCN_ERR_INVALID, "null labels");
        RCN_TRY(stage_targets(h, nullptr, labels, B, &oh, &lb));
        if (pixel_format != RCN_PIXELS_U8_ROWMAJOR && pixel_format != RCN_PIXELS_F64_COLMAJOR)
            return fail(RCN_ERR_INVALID, "unknown pixel format %d", pixel_format);
        if (!images) return fail(RCN_ERR_INVALID, "null images");
        StagedIn in;
        RCN_TRY(in.stage(images, B * H * W * pixel_bytes(pixel_format), h->in_stage, h->stream, nullptr));
        RCN_TRY(accumulate_images_dev(h, in.dev, pixel_format, lb, B, H, W, nullptr, req, done));
    } else {
        RCN_TRY(accumulate_dev(h, nullptr, nullptr, nullptr, 0, nullptr, req, done));
    }
    if (B && (!is_device_ptr(images) || !is_device_ptr(labels))) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int rcn_cuda_accumulate_gradients(rcn_cuda_handle h, const double* feats, const double* onehot, const int64_t* labels,
                                  size_t B) {
    RCN_ENTER(h);
    return accumulate_gradients(h, feats, onehot, labels, B, StepRequest{}, nullptr);
}

int rcn_cuda_accumulate_gradients_images(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                                         size_t B, size_t H, size_t W) {
    RCN_ENTER(h);
    return accumulate_gradients_images(h, images, pixel_format, labels, B, H, W, StepRequest{}, nullptr);
}

int rcn_cuda_apply_gradients(rcn_cuda_handle h, double eta, size_t batch) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (batch == 0) return RCN_OK;  // chunks_exact never yields an empty batch (rcn.rs:147)
    // (eta / batch.len() as f64)  (rcn.rs:214); on a group the exchange over NVLink peer memory fused with the update (dp.cu)
    return finish_step(h, step_update(h, eta / (double)batch), StepDone::nothing);
}

// Every entry point that drains the model's stream ends the hazard x_owns_cursor guards against.
static void stream_drained(rcn_cuda_model* h) { h->x_owns_cursor = false; }

// One training step: the fused small-network path lets kernel B apply the update (one GPU) or push the gradients to the
// peers; finish_step launches whatever it left.  On a connected data-parallel group B is this rank's shard and the update
// uses the global batch (rcn.rs:214).
int rcn_cuda_train_batch(rcn_cuda_handle h, const double* feats, const double* onehot, const int64_t* labels, size_t B,
                         double eta) {
    RCN_ENTER(h);
    if (B == 0) return accumulate_gradients(h, feats, onehot, labels, 0, StepRequest{}, nullptr);
    const StepRequest req{step_update(h, eta / (double)(B * (size_t)(h->dp.connected ? h->dp.world : 1)))};
    StepDone done;
    RCN_TRY(accumulate_gradients(h, feats, onehot, labels, B, req, &done));
    return finish_step(h, req.upd, done);
}

int rcn_cuda_train_batch_images(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                                size_t H, size_t W, double eta) {
    RCN_ENTER(h);
    if (B == 0) return accumulate_gradients_images(h, images, pixel_format, labels, 0, H, W, StepRequest{}, nullptr);
    const StepRequest req{step_update(h, eta / (double)(B * (size_t)(h->dp.connected ? h->dp.world : 1)))};
    StepDone done;
    RCN_TRY(accumulate_gradients_images(h, images, pixel_format, labels, B, H, W, req, &done));
    return finish_step(h, req.upd, done);
}

int rcn_cuda_last_batch_stats(rcn_cuda_handle h, double* cost, uint64_t* hits) {
    RCN_ENTER(h);
    if (!h->stats_valid) return fail(RCN_ERR_STATE, "no batch has been accumulated yet");
    double host[2];
    RCN_CUDA_TRY(cudaMemcpyAsync(host, h->small.p, sizeof(host), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (cost) *cost = host[0];
    if (hits) memcpy(hits, &host[1], sizeof(uint64_t));
    return RCN_OK;
}

// ---- epoch mode: rcn.rs:144-149 over a dataset resident in device memory ---------------------------------------------
int rcn_cuda_epoch_bind(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                        const int64_t* perm, size_t n_samples, size_t H, size_t W, size_t B) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!images || !labels || B == 0 || n_samples < B) return fail(RCN_ERR_INVALID, "epoch_bind needs images, labels and n_samples >= B > 0");
    if (!is_device_ptr(images) || !is_device_ptr(labels) || (perm && !is_device_ptr(perm)))
        return fail(RCN_ERR_INVALID, "epoch mode needs a dataset resident in device memory");
    if (pixel_format != RCN_PIXELS_U8_ROWMAJOR && pixel_format != RCN_PIXELS_F64_COLMAJOR)
        return fail(RCN_ERR_INVALID, "unknown pixel format %d", pixel_format);
    RCN_TRY(ensure_plan(h, H, W));
    RCN_TRY(check_feature_width(h, h->plan.L));
    RCN_TRY(h->ep_state.reserve((kEpSlots + B) * sizeof(int64_t)));
    RCN_CUDA_TRY(cudaMemsetAsync(h->ep_state.p, 0, (kEpSlots + B) * sizeof(int64_t), h->stream));
    RCN_TRY(h->feats.reserve(h->plan.L * B * sizeof(double)));
    h->ep_images = images; h->ep_labels = labels; h->ep_perm = perm; h->ep_fmt = pixel_format;
    h->ep_n = n_samples; h->ep_H = H; h->ep_W = W; h->ep_B = B;
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));   // the cursor is zero before any step kernel can look at it
    stream_drained(h);
    return RCN_OK;
}

int rcn_cuda_epoch_seek(rcn_cuda_handle h, size_t position) {
    RCN_ENTER(h);
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_epoch_bind first");
    if (position + h->ep_B > h->ep_n) return fail(RCN_ERR_INVALID, "position %zu leaves fewer than B samples", position);
    const long long pos = (long long)position;
    RCN_CUDA_TRY(cudaMemcpyAsync(h->ep_state.p, &pos, sizeof(pos), cudaMemcpyHostToDevice, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    return RCN_OK;
}

int rcn_cuda_epoch_position(rcn_cuda_handle h, size_t* position) {
    RCN_ENTER(h);
    if (!h->ep_images || !position) return fail(RCN_ERR_STATE, "no dataset bound / null output");
    long long pos = 0;
    RCN_CUDA_TRY(cudaMemcpyAsync(&pos, h->ep_state.p, sizeof(pos), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    *position = (size_t)pos;
    return RCN_OK;
}

// The update of a step over the bound dataset: it also advances the device-side cursor.
static SnUpdate epoch_update(rcn_cuda_model* h, double scale) {
    return step_update(h, scale, h->ep_state.as<long long>(), (long long)h->ep_B, (long long)h->ep_n);
}

static int epoch_accumulate(rcn_cuda_model* h, const StepRequest& req, StepDone* done) {
    RCN_TRY(require_params(h));
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_epoch_bind first");
    BatchIndex bi;
    bi.cursor = h->ep_state.as<long long>();
    bi.perm = (const long long*)h->ep_perm;
    bi.labels_all = (const long long*)h->ep_labels;
    bi.labels_batch = h->ep_state.as<long long>() + kEpSlots;
    bi.batch = (long long)h->ep_B;   // lets kernel A ask L2 for the next step's images (smallnet.cu)
    bi.n_samples = (long long)h->ep_n;
    return accumulate_images_dev(h, h->ep_images, h->ep_fmt, nullptr, h->ep_B, h->ep_H, h->ep_W, &bi, req, done);
}

int rcn_cuda_epoch_accumulate(rcn_cuda_handle h) {
    RCN_ENTER(h);
    return epoch_accumulate(h, StepRequest{}, nullptr);
}

int rcn_cuda_epoch_apply(rcn_cuda_handle h, double eta, size_t global_batch) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_epoch_bind first");
    if (global_batch == 0) return fail(RCN_ERR_INVALID, "global batch is zero");
    return finish_step(h, epoch_update(h, eta / (double)global_batch), StepDone::nothing);
}

int rcn_cuda_epoch_step(rcn_cuda_handle h, double eta) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_epoch_bind first");
    const StepRequest req{epoch_update(h, eta / (double)(h->ep_B * (size_t)(h->dp.connected ? h->dp.world : 1)))};
    StepDone done;
    RCN_TRY(epoch_accumulate(h, req, &done));
    return finish_step(h, req.upd, done);
}

int rcn_cuda_epoch_run(rcn_cuda_handle h, double eta, size_t n_steps) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_epoch_bind first");
    if (n_steps > (size_t)1 << 30) return fail(RCN_ERR_INVALID, "too many steps in one call");
    for (size_t k = 0; k < n_steps; ++k) RCN_TRY(rcn_cuda_epoch_step(h, eta));
    return RCN_OK;
}

// ---- pipelined loop over a HOST-resident dataset: rcn.rs:147-149 ------------------------------------------------------
// Streamed loop over the epoch's labels in tgt_stage: the copy engine streams the pinned u8 images into the device ring while
// earlier chunks train, kernel B writes each step's result into pinned host memory, and the host launches CUDA graphs of
// several steps each and queues the copies.
static int train_epoch_streamed(rcn_cuda_model* h, const void* images, size_t n_steps, size_t H, size_t W, size_t B, double scale) {
    HostEpoch& ep = h->host_epoch;
    const size_t img_bytes = B * H * W;
    const size_t spg = (size_t)hs_steps_per_graph();
    // The epoch as a sequence of graph launches: as many `spg`-step graphs as fit, then the largest of 20 / 10 / 5 / 2 / 1 steps
    // that still fits -- as few launches as possible: with copies on the link a graph boundary costs 4-5 us and now and then
    // 27 us (a short FIRST graph to get going sooner measured worse for that reason: 507-519 us against 479 for a 20-step
    // epoch; its launch latency passes while the first chunk crosses the link anyway).
    std::vector<int> plan_g;
    for (size_t left = n_steps; left;) {
        size_t g = 1;
        if (left >= spg) g = spg;
        else
            for (size_t c : {(size_t)20, (size_t)10, (size_t)5, (size_t)2})
                if (c < spg && left >= c) { g = c; break; }
        plan_g.push_back((int)g);
        left -= g;
    }
    RCN_TRY(ep.state.reserve((kHsStateSlots + B) * sizeof(long long)));
    RCN_TRY(h->feats.reserve(h->plan.L * B * sizeof(double)));
    long long* st = ep.state.as<long long>();
    BatchIndex bi;
    bi.cursor = st;
    bi.labels_all = h->tgt_stage.as<long long>();
    bi.labels_batch = st + kHsStateSlots;
    bi.window = (long long)(kHsRingSteps * B);
    bi.arrived = st + 3;
    // cursor and arrival counter start at zero; after that graph replays
    const long long init[kHsStateSlots] = {};
    RCN_CUDA_TRY(cudaMemcpyAsync(st, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
    HostEpoch::Key key;   // the graphs do not depend on the epoch length
    key.B = B; key.H = H; key.W = W; key.scale = scale;
    key.labels = h->tgt_stage.p;   // (grows with the epoch length: a longer epoch than any before re-captures)
    key.alloc_gen = alloc_generation().load(std::memory_order_relaxed);
    memcpy(&key.mean_bits, &h->mean, sizeof(double));   // a set_scale / gen_scales since the capture re-captures
    memcpy(&key.sd_bits, &h->sd, sizeof(double));
    key.stats = ep.stats.p; key.ring = ep.ring.p; key.state = st; key.grads = h->grads; key.stream = h->stream;
    key.dp = h->dp.connected;
    key.window = bi.window;
    if (ep.graphs.empty() || !(key == ep.key)) {
        for (auto& kv : ep.graphs) cudaGraphExecDestroy(kv.second);
        ep.graphs.clear();
        // warm-up outside capture: reserves every scratch buffer and sets kernel attributes (no parameter update, no push to
        // the peers)
        BatchIndex bi_warm = bi;
        bi_warm.arrived = nullptr;   // nothing has been copied yet: the warm-up trains on whatever the ring holds
        StepRequest warm;
        warm.push = false;
        RCN_TRY(accumulate_images_dev(h, ep.ring.p, RCN_PIXELS_U8_ROWMAJOR, nullptr, B, H, W, &bi_warm, warm));
        RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
        key.alloc_gen = alloc_generation().load(std::memory_order_relaxed);   // the warm-up may have grown scratch buffers
        ep.key = key;
    }
    // `g` consecutive steps in ONE graph: a step is only tens of microseconds long, so the host's per-launch cost is spread
    // over several of them; the remainder of the epoch replays the one-step graph.
    auto capture_steps = [&](int g, cudaGraphExec_t* out) -> int {
        cudaGraph_t graph = nullptr;
        RCN_CUDA_TRY(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        int rc = RCN_OK;
        const StepRequest req{step_update(h, scale, st, (long long)B, kHsNoWrap, ep.stats.p, true)};
        for (int q = 0; q < g && rc == RCN_OK; ++q) {
            StepDone done;
            rc = accumulate_images_dev(h, ep.ring.p, RCN_PIXELS_U8_ROWMAJOR, nullptr, B, H, W, &bi, req, &done);
            if (rc == RCN_OK) rc = finish_step(h, req.upd, done);
        }
        cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
        if (rc != RCN_OK) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); return rc; }
        if (ce != cudaSuccess || !graph) return fail(RCN_ERR_CUDA, "stream capture of the training step failed: %s", cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(out, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { *out = nullptr; return fail(RCN_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
        return RCN_OK;
    };
    for (int g : plan_g) {
        if (ep.graphs.count(g)) continue;
        cudaGraphExec_t ge = nullptr;
        RCN_TRY(capture_steps(g, &ge));
        ep.graphs[g] = ge;
    }
    // Copies first (the driver queues them; each waits on the device for its ring slots), then the graph launches.
    const StreamMemOps& mo = stream_mem_ops(h->device);
    const CUdeviceptr cursor_dev = (CUdeviceptr)reinterpret_cast<uintptr_t>(st);
    const char* src = static_cast<const char*>(images);
    RCN_TRY(ep.counts.reserve(n_steps));
    // the state block (cursor 0, arrived 0) must be in place before the first counter copy can land
    RCN_CUDA_TRY(cudaEventRecord(ep.fork, h->stream));
    RCN_CUDA_TRY(cudaStreamWaitEvent(ep.flag_stream, ep.fork, 0));
    size_t a = 0, k = 0, n_copy = 0;
    auto enqueue_copy = [&]() -> int {
        // ramp: while the copies are only a few chunks ahead of the training steps a long copy would hold back the steps
        // waiting for its first chunk (the counter moves when a copy has landed completely)
        size_t g = a < 2 ? 1 : (a < 16 ? 2 : (a < 32 ? 4 : kHsMaxCopy));
        g = std::min(g, n_steps - a);
        g = std::min(g, kHsQuarter - a % kHsQuarter);                      // never across a quarter of the ring
        if (a >= kHsRingSteps && a % kHsQuarter == 0) {
            // entering a quarter whose slots held steps [a - ring, a + quarter - ring): all of them must have trained
            if (mo.wait64(ep.copy_stream, cursor_dev, (cuuint64_t)((a + kHsQuarter - kHsRingSteps) * B), CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
                return fail(RCN_ERR_CUDA, "cuStreamWaitValue64 failed");
        }
        RCN_CUDA_TRY(cudaMemcpyAsync(ep.ring.as<char>() + (a % kHsRingSteps) * img_bytes, src + a * img_bytes, g * img_bytes,
                                     cudaMemcpyHostToDevice, ep.copy_stream));
        a += g;
        ep.counts.p[n_copy] = (long long)(a * B);
        cudaEvent_t ev = ep.ev_arrived[n_copy % kHsEvents];
        RCN_CUDA_TRY(cudaEventRecord(ev, ep.copy_stream));
        RCN_CUDA_TRY(cudaStreamWaitEvent(ep.flag_stream, ev, 0));
        // (cuStreamWriteValue64 here instead measured the same: 476 vs 478 us for a 20-step epoch)
        RCN_CUDA_TRY(cudaMemcpyAsync(st + 3, ep.counts.p + n_copy, sizeof(long long), cudaMemcpyHostToDevice, ep.flag_stream));
        ++n_copy;
        return RCN_OK;
    };
    // One chunk's copy, then the first graph launch (its launch latency passes while the chunk crosses the link; kernel A
    // waits on the device for whatever has not arrived yet), then copies and launches interleaved, the copies enqueued half a
    // ring ahead of the launches.
    RCN_TRY(enqueue_copy());
    for (int g : plan_g) {
        RCN_CUDA_TRY(cudaGraphLaunch(ep.graphs[g], h->stream));
        k += (size_t)g;
        while (a < n_steps && a < k + kHsRingSteps / 2) RCN_TRY(enqueue_copy());
    }
    // A + B (+ exchange/update) per replayed step
    g_launches.fetch_add((unsigned long long)n_steps * (2 + (h->dp.connected ? 1 : 0)), std::memory_order_relaxed);
    return RCN_OK;
}

// General loop over the epoch's labels in tgt_stage: double-buffered cudaMemcpyAsync of each step's images on the copy stream.
static int train_epoch_buffered(rcn_cuda_model* h, const void* images, int pixel_format, size_t n_steps, size_t H, size_t W,
                                size_t B, double scale) {
    HostEpoch& ep = h->host_epoch;
    const size_t img_bytes = B * H * W * pixel_bytes(pixel_format);
    for (DevBuf& buf : ep.host_slot) RCN_TRY(buf.reserve(img_bytes));
    const int64_t* labels_dev = h->tgt_stage.as<int64_t>();
    // everything the previous user of the staging slots enqueued on the compute stream must be finished first
    RCN_CUDA_TRY(cudaEventRecord(ep.ev_consumed[0], h->stream));
    RCN_CUDA_TRY(cudaEventRecord(ep.ev_consumed[1], h->stream));
    // unarmed: kernel B leaves the update to the update kernel (or the exchange kernel)
    const SnUpdate update = step_update(h, scale);
    const char* img = (const char*)images;
    for (size_t k = 0; k < n_steps; ++k) {
        const int slot = (int)(k & 1);
        char* dst = ep.host_slot[slot].as<char>();
        // H2D of chunk k on the copy stream: overlaps the kernels of chunk k-1
        RCN_CUDA_TRY(cudaStreamWaitEvent(ep.copy_stream, ep.ev_consumed[slot], 0));
        RCN_CUDA_TRY(cudaMemcpyAsync(dst, img + k * img_bytes, img_bytes, cudaMemcpyHostToDevice, ep.copy_stream));
        RCN_CUDA_TRY(cudaEventRecord(ep.ev_copied[slot], ep.copy_stream));
        RCN_CUDA_TRY(cudaStreamWaitEvent(h->stream, ep.ev_copied[slot], 0));
        RCN_TRY(accumulate_images_dev(h, dst, pixel_format, labels_dev + k * B, B, H, W, nullptr));
        RCN_CUDA_TRY(cudaEventRecord(ep.ev_consumed[slot], h->stream));
        RCN_TRY(finish_step(h, update, StepDone::nothing));
        // D2H of this step's result (cost, hits evaluated with the pre-update parameters)
        RCN_CUDA_TRY(cudaMemcpyAsync(ep.stats.p + 2 * k, h->small.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    RCN_CUDA_TRY(cudaStreamSynchronize(ep.copy_stream));
    return RCN_OK;
}

int rcn_cuda_train_epoch_host(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                              size_t n_samples, size_t H, size_t W, size_t B, double eta, size_t global_batch,
                              double* cost_out, uint64_t* hits_out, size_t* n_steps_out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n_steps_out) *n_steps_out = 0;
    if (B == 0) return fail(RCN_ERR_INVALID, "batch size is zero");
    if (pixel_format != RCN_PIXELS_U8_ROWMAJOR && pixel_format != RCN_PIXELS_F64_COLMAJOR)
        return fail(RCN_ERR_INVALID, "unknown pixel format %d", pixel_format);
    const size_t n_steps = n_samples / B;       // chunks_exact: the remainder is dropped (rcn.rs:147)
    if (n_steps == 0) return RCN_OK;
    if (!images || !labels) return fail(RCN_ERR_INVALID, "null images / labels");
    if (is_device_ptr(images) || is_device_ptr(labels))
        return fail(RCN_ERR_INVALID, "train_epoch_host takes HOST buffers; use rcn_cuda_epoch_bind for a device-resident dataset");
    RCN_TRY(ensure_plan(h, H, W));
    RCN_TRY(check_feature_width(h, h->plan.L));
    if (global_batch == 0) global_batch = B * (size_t)(h->dp.connected ? h->dp.world : 1);
    const size_t img_bytes = B * H * W * pixel_bytes(pixel_format);
    HostEpoch& ep = h->host_epoch;
    RCN_TRY(ep.setup());
    RCN_TRY(ep.stats.reserve(2 * n_steps));
    // The streamed loop needs a pinned, 16-byte aligned u8 dataset, steps that run kernel A with the staged front end on the
    // ring (its image-loading lanes wait for the arrival counter), 64-bit stream memory operations (the copy stream's wait for
    // free ring slots) and a compute stream that is not being captured.  (No ring for a network kernel A does not train.)
    bool streamed = false;
    if (pixel_format == RCN_PIXELS_U8_ROWMAJOR && h->use_small && B <= smallnet_max_batch() && img_bytes % 16 == 0 &&
        (reinterpret_cast<uintptr_t>(images) & 15) == 0 && is_pinned_host_ptr(images) && kHsRingSteps * B < (1ull << 31) &&
        stream_mem_ops(h->device).ok) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        RCN_CUDA_TRY(cudaStreamIsCapturing(h->stream, &cs));
        if (cs == cudaStreamCaptureStatusNone) {
            RCN_TRY(ep.ring.reserve(kHsRingSteps * img_bytes));
            SmallNetFront fr;
            streamed = fused_front(h, ep.ring.p, pixel_format, H, W, nullptr, &fr) && fr.use_cp;
        }
    }
    // The legacy default stream cannot be captured: the streamed loop runs on the model's own stream, ordered after whatever
    // the caller has enqueued on the legacy stream; the call drains that stream before it returns.
    struct StreamSwap {
        rcn_cuda_model* m; cudaStream_t saved;
        StreamSwap(rcn_cuda_model* m_) : m(m_), saved(m_->stream) {}
        ~StreamSwap() { m->stream = saved; }
    } swap_guard(h);
    if (streamed && h->stream == nullptr) {
        RCN_CUDA_TRY(cudaEventRecord(ep.fork, nullptr));
        RCN_CUDA_TRY(cudaStreamWaitEvent(h->own_stream, ep.fork, 0));
        h->stream = h->own_stream;
    }
    // the labels of the whole epoch go up in ONE copy (one driver call per step less); images stream chunk by chunk
    RCN_TRY(h->tgt_stage.reserve(n_steps * B * sizeof(int64_t)));
    RCN_CUDA_TRY(cudaMemcpyAsync(h->tgt_stage.p, labels, n_steps * B * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    const double scale = eta / (double)global_batch;   // (eta / batch.len() as f64)  (rcn.rs:214)
    RCN_TRY(streamed ? train_epoch_streamed(h, images, n_steps, H, W, B, scale)
                     : train_epoch_buffered(h, images, pixel_format, n_steps, H, W, B, scale));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    for (size_t k = 0; k < n_steps; ++k) {
        if (cost_out) cost_out[k] = ep.stats.p[2 * k];
        if (hits_out) memcpy(&hits_out[k], &ep.stats.p[2 * k + 1], sizeof(uint64_t));
    }
    h->stats_valid = true;
    h->last_B = B;
    if (n_steps_out) *n_steps_out = n_steps;
    return RCN_OK;
}

// ---- data-parallel group (dp.cu) -------------------------------------------------------------------------------------
int rcn_cuda_dp_init(rcn_cuda_handle h, int world, int rank, void* ipc_handle_out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    RCN_TRY(dp_alloc(h->dp, world, rank, h->n_params, h->stream));
    if (ipc_handle_out) {
        cudaIpcMemHandle_t hd;
        RCN_CUDA_TRY(cudaIpcGetMemHandle(&hd, h->dp.block));
        static_assert(sizeof(hd) == 64, "cudaIpcMemHandle_t is 64 bytes");
        memcpy(ipc_handle_out, &hd, sizeof(hd));
    }
    return RCN_OK;
}

int rcn_cuda_dp_connect_ipc(rcn_cuda_handle h, const void* all_handles) {
    RCN_ENTER(h);
    if (!h->dp.block) return fail(RCN_ERR_STATE, "call rcn_cuda_dp_init first");
    if (!all_handles) return fail(RCN_ERR_INVALID, "null handles");
    for (int q = 0; q < h->dp.world; ++q) {
        if (q == h->dp.rank) continue;
        cudaIpcMemHandle_t hd;
        memcpy(&hd, (const char*)all_handles + (size_t)q * sizeof(hd), sizeof(hd));
        void* p = nullptr;
        RCN_CUDA_TRY(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
        h->dp.peers[q] = p; h->dp.imported[q] = true;
    }
    h->dp.connected = h->dp.world > 1;
    return RCN_OK;
}

int rcn_cuda_dp_connect_local(rcn_cuda_handle h, const rcn_cuda_handle* group) {
    RCN_ENTER(h);
    if (!h->dp.block) return fail(RCN_ERR_STATE, "call rcn_cuda_dp_init first");
    if (!group) return fail(RCN_ERR_INVALID, "null group");
    for (int q = 0; q < h->dp.world; ++q) {
        if (q == h->dp.rank) continue;
        rcn_cuda_model* o = group[q];
        if (!o || !o->dp.block || o->dp.world != h->dp.world || o->dp.rank != q || o->dp.n != h->dp.n)
            return fail(RCN_ERR_INVALID, "group member %d is not an initialised rank %d of a %d-rank group with %zu parameters", q, q,
                        h->dp.world, h->dp.n);
        if (o->device != h->device) {
            int can = 0;
            RCN_CUDA_TRY(cudaDeviceCanAccessPeer(&can, h->device, o->device));
            if (!can) return fail(RCN_ERR_CUDA, "device %d cannot access device %d as a peer", h->device, o->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return fail(RCN_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) failed: %s", o->device, cudaGetErrorString(e));
            cudaGetLastError();
        }
        h->dp.peers[q] = o->dp.block; h->dp.imported[q] = false;
    }
    h->dp.connected = h->dp.world > 1;
    return RCN_OK;
}

int rcn_cuda_dp_shutdown(rcn_cuda_handle h) {
    RCN_ENTER(h);
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    dp_release(h->dp);
    h->dp_pushed = false;
    return RCN_OK;
}

static int timeline_reset(rcn_cuda_model* h) {
    static Timeline init;   // 4.3 KB: too large for the stack of a small thread
    memset(&init, 0, sizeof(init));
    memset(init.t0, 0xff, sizeof(init.t0));
    RCN_CUDA_TRY(cudaMemcpyAsync(h->timeline.p, &init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int rcn_cuda_timeline_enable(rcn_cuda_handle h, int on) {
    RCN_ENTER(h);
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    if (on) {
        RCN_TRY(h->timeline.reserve(sizeof(Timeline)));
        RCN_TRY(timeline_reset(h));
    }
    if ((on != 0) != h->tl_on) alloc_generation().fetch_add(1, std::memory_order_relaxed);   // captured steps hold the pointer by value
    h->tl_on = on != 0;
    h->small_desc.tl = h->tl_on ? h->timeline.as<Timeline>() : nullptr;
    return RCN_OK;
}

int rcn_cuda_timeline_read(rcn_cuda_handle h, uint64_t* stamps, uint32_t* launches) {
    RCN_ENTER(h);
    if (!h->tl_on) return fail(RCN_ERR_STATE, "the timeline is not enabled");
    if (!stamps || !launches) return fail(RCN_ERR_INVALID, "null output");
    static Timeline host;
    RCN_CUDA_TRY(cudaMemcpyAsync(&host, h->timeline.p, sizeof(host), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    stream_drained(h);
    memcpy(stamps, host.t0, sizeof(host.t0));
    memcpy(stamps + kTlKernels * kTlRing, host.t1, sizeof(host.t1));
    for (int k = 0; k < kTlKernels; ++k) launches[k] = host.seq[k];
    return RCN_OK;
}

int rcn_cuda_dp_error(rcn_cuda_handle h, int* error) {
    RCN_ENTER(h);
    if (!error) return fail(RCN_ERR_INVALID, "null output");
    unsigned e = 0;
    RCN_TRY(dp_read_error(h->dp, h->stream, &e));
    stream_drained(h);
    *error = (int)e;
    if (e) return fail(RCN_ERR_STATE, "data-parallel group: a gradient exchange timed out waiting for a peer (a rank died, raised before "
                                      "its launch, or ran a different number of steps); the parameters of this replica are NaN");
    return RCN_OK;
}

int rcn_cuda_bind_gradient_buffer(rcn_cuda_handle h, double* device_ptr, size_t n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (!device_ptr) {
        RCN_TRY(h->grads_own.reserve(h->n_params * sizeof(double)));
        h->grads = h->grads_own.as<double>();
        h->grads_bound = false;
        return RCN_OK;
    }
    if (n != h->n_params) return fail(RCN_ERR_SHAPE, "gradient buffer must hold %zu doubles, got %zu", h->n_params, n);
    if (!is_device_ptr(device_ptr)) return fail(RCN_ERR_INVALID, "gradient buffer must be device memory");
    h->grads = device_ptr;
    h->grads_bound = true;
    return RCN_OK;
}

int rcn_cuda_gradient_buffer(rcn_cuda_handle h, double** device_ptr, size_t* n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (device_ptr) *device_ptr = h->grads;
    if (n) *n = h->n_params;
    return RCN_OK;
}

int rcn_cuda_get_gradients(rcn_cuda_handle h, double* flat, size_t n) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (n != h->n_params || !flat) return fail(RCN_ERR_SHAPE, "model has %zu parameters, got %zu", h->n_params, n);
    return deliver(h, flat, h->grads, n * sizeof(double));
}

int rcn_cuda_get_activations(rcn_cuda_handle h, size_t layer, double* out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size() || !out) return fail(RCN_ERR_INVALID, "bad layer / null destination");
    if (!h->last_B) return fail(RCN_ERR_STATE, "no batch has been accumulated yet");
    return deliver(h, out, h->act(layer, h->last_B), h->rows[layer] * h->last_B * sizeof(double));
}

int rcn_cuda_get_deltas(rcn_cuda_handle h, size_t layer, double* out) {
    RCN_ENTER(h);
    RCN_TRY(require_params(h));
    if (layer >= h->rows.size() || !out) return fail(RCN_ERR_INVALID, "bad layer / null destination");
    if (!h->last_B) return fail(RCN_ERR_STATE, "no batch has been accumulated yet");
    return deliver(h, out, h->delta(layer, h->last_B), h->rows[layer] * h->last_B * sizeof(double));
}

// ---- launch accounting ------------------------------------------------------------------------------
int rcn_cuda_kernel_launches(uint64_t* count) {
    if (!count) return fail(RCN_ERR_INVALID, "null count");
    *count = g_launches.load();
    return RCN_OK;
}

int rcn_cuda_allocation_generation(uint64_t* generation) {
    if (!generation) return fail(RCN_ERR_INVALID, "null generation");
    *generation = alloc_generation().load(std::memory_order_relaxed);
    return RCN_OK;
}

int rcn_cuda_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (on) {
        for (auto& r : g_prof) { cudaEventDestroy(r.start); cudaEventDestroy(r.stop); }
        g_prof.clear();
    }
    g_profiling.store(on != 0);
    return RCN_OK;
}

int rcn_cuda_profile_report(char* json_out, size_t capacity) {
    if (!json_out || capacity < 3) return fail(RCN_ERR_INVALID, "report buffer too small");
    RCN_CUDA_TRY(cudaDeviceSynchronize());
    std::map<std::string, std::pair<unsigned long long, double>> agg;
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        for (auto& r : g_prof) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, r.start, r.stop) != cudaSuccess) { cudaGetLastError(); continue; }
            auto& a = agg[r.name];
            a.first += 1; a.second += ms;
        }
    }
    std::string js = "{";
    bool first = true;
    for (auto& kv : agg) {
        char buf[256];
        snprintf(buf, sizeof(buf), "%s\"%s\": {\"launches\": %llu, \"total_ms\": %.6f}", first ? "" : ", ", kv.first.c_str(),
                 kv.second.first, kv.second.second);
        js += buf;
        first = false;
    }
    js += "}";
    if (js.size() + 1 > capacity) return fail(RCN_ERR_INVALID, "report needs %zu bytes", js.size() + 1);
    memcpy(json_out, js.c_str(), js.size() + 1);
    return RCN_OK;
}

// ---- op-level API ---------------------------------------------------------------------------------

int rcn_cuda_convolve_2d(int device, void* cuda_stream, const double* m, size_t H, size_t W, const double* kernel,
                         size_t kh, size_t kw, int padding, double* out) {
    if (!m || !kernel || !out) return fail(RCN_ERR_INVALID, "null pointer");
    if (padding != RCN_PADDING_NONE && padding != RCN_PADDING_SAME) return fail(RCN_ERR_INVALID, "unknown padding %d", padding);
    // kernel.rs:123-128
    if ((kh == 0 && kw == 0) || kh > H || kw > W || kh == 0 || kw == 0)
        return fail(RCN_ERR_SHAPE, "convolve_2d expects 'self.shape() >= kernel_shape() > 0', received (%zu, %zu) and (%zu, %zu) respectively.", H, W, kh, kw);
    // kernel.rs:131-135
    if ((kh % 2 == 0 || kw % 2 == 0) && padding == RCN_PADDING_SAME)
        return fail(RCN_ERR_SHAPE, "convolve_2d expects kernel dimensions to be odd when padding mode set to 'SAME', got (%zu, %zu)", kh, kw);
    // kernel.rs:154-158: the padded copy indexes self[(cy-1, cx-1)] up to cy = H + kh/2 - 1 => out of bounds for kh/2 >= 2
    if (padding == RCN_PADDING_SAME && (kh / 2 >= 2 || kw / 2 >= 2))
        return fail(RCN_ERR_OUT_OF_BOUNDS, "Matrix index out of bounds. (SAME padding with a (%zu, %zu) kernel, kernel.rs:156)", kh, kw);
    if (H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "matrix too large");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const bool same = padding == RCN_PADDING_SAME;
    const size_t on = same ? H * W : (H - kh + 1) * (W - kw + 1);
    const void *m_dev = nullptr, *k_dev = nullptr; void* o_dev = nullptr; bool host = false;
    RCN_TRY(c.in(m, H * W * 8, tl_op_in, &m_dev));
    RCN_TRY(c.in(kernel, kh * kw * 8, tl_op_k, &k_dev));
    RCN_TRY(c.out(out, on * 8, tl_op_out, &o_dev, &host));
    RCN_TRY(launch_convolve_2d((const double*)m_dev, H, W, (const double*)k_dev, kh, kw, padding, (double*)o_dev, c.stream));
    return c.finish(out, o_dev, on * 8, host);
}

int rcn_cuda_convolve_2d_separated(int device, void* cuda_stream, const double* m, size_t H, size_t W, int op, int padding,
                                   double* out) {
    if (!m || !out) return fail(RCN_ERR_INVALID, "null pointer");
    if (padding != RCN_PADDING_NONE && padding != RCN_PADDING_SAME) return fail(RCN_ERR_INVALID, "unknown padding %d", padding);
    if (op < 0 || op > 3) return fail(RCN_ERR_INVALID, "unknown SeparableOperator %d", op);
    if (H < 3 || W < 3)  // kernel.rs:199-201
        return fail(RCN_ERR_SHAPE, "convolve_2d_separated expects 'self.shape() >= kernel_shape() > 0', received (%zu, %zu) and (3, 3) respectively.", H, W);
    if (H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "matrix too large");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const bool same = padding == RCN_PADDING_SAME;
    const size_t on = same ? H * W : (H - 2) * (W - 2);
    const void* m_dev = nullptr; void* o_dev = nullptr; bool host = false;
    RCN_TRY(c.in(m, H * W * 8, tl_op_in, &m_dev));
    RCN_TRY(c.out(out, on * 8, tl_op_out, &o_dev, &host));
    RCN_TRY(launch_convolve_2d_separated((const double*)m_dev, H, W, op, padding, (double*)o_dev, c.stream));
    return c.finish(out, o_dev, on * 8, host);
}

int rcn_cuda_relu(int device, void* cuda_stream, const double* m, size_t n, double* out) {
    if (n == 0) return RCN_OK;
    if (!m || !out) return fail(RCN_ERR_INVALID, "null pointer");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const void* m_dev = nullptr; void* o_dev = nullptr; bool host = false;
    RCN_TRY(c.in(m, n * 8, tl_op_in, &m_dev));
    RCN_TRY(c.out(out, n * 8, tl_op_out, &o_dev, &host));
    RCN_TRY(launch_relu((const double*)m_dev, n, (double*)o_dev, c.stream));
    return c.finish(out, o_dev, n * 8, host);
}

int rcn_cuda_pool_2d(int device, void* cuda_stream, const double* m, size_t H, size_t W, int padding, int pooling,
                     double* out, uint8_t* argmax_out) {
    if (!m || !out) return fail(RCN_ERR_INVALID, "null pointer");
    if (padding != RCN_PADDING_NONE && padding != RCN_PADDING_SAME) return fail(RCN_ERR_INVALID, "unknown padding %d", padding);
    if (pooling != RCN_POOLING_AVERAGE && pooling != RCN_POOLING_MAX) return fail(RCN_ERR_INVALID, "unknown pooling %d", pooling);
    if (H < 2 || W < 2)  // kernel.rs:246-251
        return fail(RCN_ERR_SHAPE, "stride_2d expected a matrix with dimensions greater than (2, 2), got (%zu, %zu)", H, W);
    if (pooling != RCN_POOLING_MAX) return fail(RCN_ERR_NOT_IMPLEMENTED, "Not implemented");  // kernel.rs:283-285
    if (H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "matrix too large");
    OpCtx c;
    RCN_TRY(c.enter(device, cuda_stream));
    const bool same = padding == RCN_PADDING_SAME;
    const size_t oh = same ? (H + 1) / 2 : H / 2, ow = same ? (W + 1) / 2 : W / 2;
    const size_t on = oh * ow;
    const void* m_dev = nullptr; void* o_dev = nullptr; bool host = false;
    RCN_TRY(c.in(m, H * W * 8, tl_op_in, &m_dev));
    RCN_TRY(c.out(out, on * 8, tl_op_out, &o_dev, &host));
    // aux: [int nan_flag | pad to 16 | argmax bytes]
    RCN_TRY(tl_op_aux.reserve(16 + on));
    int* flag = tl_op_aux.as<int>();
    RCN_CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), c.stream));
    uint8_t* am_dev = nullptr;
    bool am_host = false;
    if (argmax_out) {
        if (is_device_ptr(argmax_out)) am_dev = argmax_out;
        else { am_dev = tl_op_aux.as<uint8_t>() + 16; am_host = true; }
    }
    RCN_TRY(launch_pool_2d((const double*)m_dev, H, W, padding, (double*)o_dev, am_dev, flag, c.stream));
    int nan = 0;
    RCN_CUDA_TRY(cudaMemcpyAsync(&nan, flag, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    if (am_host) RCN_CUDA_TRY(cudaMemcpyAsync(argmax_out, am_dev, on, cudaMemcpyDeviceToHost, c.stream));
    if (host) RCN_CUDA_TRY(cudaMemcpyAsync(out, o_dev, on * 8, cudaMemcpyDeviceToHost, c.stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(c.stream));
    if (nan) return fail(RCN_ERR_NAN, "called `Option::unwrap()` on a `None` value (partial_cmp on NaN, kernel.rs:280)");
    return RCN_OK;
}

}  // extern "C"

// ---- the dense stack of the convolutional network handle (cnn.cuh) ------------------------------------------------
namespace rcn {

int model_evaluate_features(rcn_cuda_model* h, const double* feats, const int64_t* labels, size_t B, double* stats,
                            int64_t* labels_out) {
    RCN_TRY(require_params(h));
    if (B == 0) return RCN_OK;
    RCN_TRY(forward_dev(h, feats, B, nullptr, nullptr, false));
    const size_t n = h->rows.size();
    if (h->head == RCN_HEAD_SOFTMAX_XENT)
        return launch_softmax_xent_head(h->act(n - 1, B), h->rows[n - 1], B, labels, nullptr, labels_out, labels ? stats : nullptr,
                                        h->rs, h->stream);
    if (labels) RCN_TRY(launch_batch_stats(h->act(n - 1, B), h->rows[n - 1], B, nullptr, labels, stats, h->rs, h->stream));
    if (labels_out) RCN_TRY(launch_argmax_last(h->act(n - 1, B), h->rows[n - 1], B, labels_out, h->stream));
    return RCN_OK;
}

int model_set_head(rcn_cuda_model* h, int head) {
    if (head != RCN_HEAD_SIGMOID_QUADRATIC && head != RCN_HEAD_SOFTMAX_XENT) return fail(RCN_ERR_INVALID, "unknown head %d", head);
    if (h->params_ready) return fail(RCN_ERR_STATE, "internal: the head is set before the layer shapes");
    h->head = head;
    return RCN_OK;
}

int model_first_layer(rcn_cuda_model* h, const double** W0, const double** delta0, size_t* rows0, size_t* cols0) {
    RCN_TRY(require_params(h));
    *W0 = h->params.as<double>() + h->w_off[0];
    *delta0 = h->deltas.as<double>();
    *rows0 = h->rows[0];
    *cols0 = h->cols[0];
    return RCN_OK;
}

int model_params(rcn_cuda_model* h, double** params, size_t* n) {
    RCN_TRY(require_params(h));
    *params = h->params.as<double>();
    *n = h->n_params;
    return RCN_OK;
}

}  // namespace rcn
