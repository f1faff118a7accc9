/* rcn_cuda.h -- C ABI of librcn_cuda.so: rcn's training hot path on one B200 (sm_100a).
 *
 * The reference (jtstrader/mercer-research, crate `rcn`) has no FFI of its own; its drop-in boundary
 * is the crate's public Rust API (SURVEY.md section 8b). Each entry point below names the reference
 * item it replaces (file:line relative to /root/reference/). A Rust facade binds these 1:1
 * (rust/src/ffi.rs; INTEGRATION.md shows the `extern "C"` block and build.rs step).
 *
 * Conventions
 *  - All matrices are f64 COLUMN-MAJOR (nalgebra storage; serialization.rs:19-22 writes exactly this).
 *    A batch of B vectors of length n is an n x B column-major matrix: sample b at ptr + b*n.
 *  - Every data pointer may be a HOST or a DEVICE pointer; the library detects which
 *    (cudaPointerGetAttributes). Host buffers are staged through the model's stream and the call
 *    returns after the stream has drained; with device buffers the call only enqueues work on the
 *    model's stream (capturable into a CUDA graph once shapes have been seen once).
 *  - Every function returns an rcn_status; rcn_cuda_last_error() gives the thread-local message.
 *    Where the reference panic!()s on a contract violation the library returns RCN_ERR_SHAPE /
 *    RCN_ERR_NOT_IMPLEMENTED with the reference's message instead of aborting.
 *  - A handle is not safe for concurrent mutation (same rule as `&mut self`); distinct handles are
 *    independent. There is NO CPU fallback: without a usable CUDA device every call fails with
 *    RCN_ERR_CUDA.
 */
#ifndef RCN_CUDA_H
#define RCN_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rcn_cuda_model* rcn_cuda_handle;
typedef struct rcn_cuda_cnn* rcn_cuda_cnn_handle;

typedef enum rcn_status {
    RCN_OK = 0,
    RCN_ERR_INVALID = 1,         /* null pointer, bad enum, zero size */
    RCN_ERR_SHAPE = 2,           /* reference panics: kernel.rs:127,133,200,247; nalgebra dim mismatch */
    RCN_ERR_NOT_IMPLEMENTED = 3, /* reference panics "Not implemented": kernel.rs:284,342 (Pooling::Average in rcn's own ops) */
    RCN_ERR_CUDA = 4,            /* CUDA runtime error / no device */
    RCN_ERR_STATE = 5,           /* parameters not initialised, etc. */
    RCN_ERR_OUT_OF_BOUNDS = 6,   /* reference index panic: kernel.rs:156 (SAME padding with a >=5-wide kernel) */
    RCN_ERR_NAN = 7              /* reference panics on partial_cmp(NaN): kernel.rs:280,338 */
} rcn_status;

/* enum Padding (kernel.rs:25-28), enum Pooling (kernel.rs:32-35), enum SeparableOperator (kernel.rs:16-21):
 * values are the Rust declaration order (= bincode variant index). */
enum { RCN_PADDING_NONE = 0, RCN_PADDING_SAME = 1 };
enum { RCN_POOLING_AVERAGE = 0, RCN_POOLING_MAX = 1 };
enum { RCN_OP_TOP = 0, RCN_OP_BOTTOM = 1, RCN_OP_LEFT = 2, RCN_OP_RIGHT = 3 };
/* enum RCNLayer { Convolve2D(Padding), Pool2D(Pooling) } (rcn.rs:35-38), flattened. */
enum { RCN_LAYER_CONV_NONE = 0, RCN_LAYER_CONV_SAME = 1, RCN_LAYER_POOL_AVERAGE = 2, RCN_LAYER_POOL_MAX = 3 };
/* Pixel formats accepted by the image entry points. */
enum {
    RCN_PIXELS_U8_ROWMAJOR = 0,  /* `image` crate GrayImage buffer, before get_pixel_matrix (lib.rs:27-33) */
    RCN_PIXELS_F64_COLMAJOR = 1, /* DMatrix<f64> H x W as get_pixel_matrix returns it */
    RCN_PIXELS_F64_NHWC = 2      /* f64 (B, H, W, C) channels-last; only the rcn_cuda_cnn_* entry points accept it */
};

const char* rcn_cuda_last_error(void);
int rcn_cuda_version(void);
int rcn_cuda_device_count(int* count);

/* ---- model lifetime: RCN::new (rcn.rs:58-75) -------------------------------------------------- */
int rcn_cuda_create(size_t classes, const int32_t* convpool_cfg, size_t n_convpool,
                    const size_t* feedforward_cfg, size_t n_feedforward, int device,
                    rcn_cuda_handle* out);
int rcn_cuda_destroy(rcn_cuda_handle h);
/* Run on an existing cudaStream_t (e.g. torch's current stream). NULL is the CUDA legacy default stream (what
 * torch hands out as its default stream); RCN_STREAM_OWN restores the model's private non-blocking stream. */
#define RCN_STREAM_OWN ((void*)(intptr_t)-1)
int rcn_cuda_set_stream(rcn_cuda_handle h, void* cuda_stream);
int rcn_cuda_synchronize(rcn_cuda_handle h);

/* ---- shapes ------------------------------------------------------------------------------------ */
/* Geometry walk of flatten_feature_set (rcn.rs:317-356): number of maps and their size. */
int rcn_cuda_feature_shape(rcn_cuda_handle h, size_t H, size_t W, size_t* n_maps, size_t* map_h, size_t* map_w);
/* load_weights_and_bias (rcn.rs:425-457): allocates zeroed W_l (rows x cols) and b_l with the reference's
 * shapes, including its `4^c / 2^p * l` first-layer width. Values are then injected with set_params
 * (the reference draws them from an unseeded thread_rng, rcn.rs:500-523). */
int rcn_cuda_init_params(rcn_cuda_handle h, size_t feature_len);
/* Explicit layer shapes (rows[i] x cols[i], cols[i] == rows[i-1]) for a model restored from a bincode checkpoint
 * (bincode::deserialize, main.rs:50 / backend/src/main.rs:68): the file, not the config, decides the matrices. */
int rcn_cuda_init_params_shapes(rcn_cuda_handle h, const size_t* rows, const size_t* cols, size_t n_layers);
int rcn_cuda_num_layers(rcn_cuda_handle h, size_t* n_layers);
int rcn_cuda_layer_shape(rcn_cuda_handle h, size_t layer, size_t* rows, size_t* cols);
int rcn_cuda_param_count(rcn_cuda_handle h, size_t* n);

/* ---- parameters: Weights / Bias (rcn.rs:28-31; layout of serialization.rs:16-24,109-113) ------ */
int rcn_cuda_set_weights(rcn_cuda_handle h, size_t layer, size_t rows, size_t cols, const double* w);
int rcn_cuda_get_weights(rcn_cuda_handle h, size_t layer, double* w);
int rcn_cuda_set_bias(rcn_cuda_handle h, size_t layer, size_t n, const double* b);
int rcn_cuda_get_bias(rcn_cuda_handle h, size_t layer, double* b);
/* Whole model as one flat buffer [W0|b0|W1|b1|...]. */
int rcn_cuda_set_params(rcn_cuda_handle h, const double* flat, size_t n);
int rcn_cuda_get_params(rcn_cuda_handle h, double* flat, size_t n);
/* scale_set (rcn.rs:21): (mean, sd) used by the standardise step. */
int rcn_cuda_set_scale(rcn_cuda_handle h, double mean, double sd);
int rcn_cuda_get_scale(rcn_cuda_handle h, double* mean, double* sd);

/* ---- feature stage ----------------------------------------------------------------------------- */
/* flatten_feature_set (rcn.rs:317-356) over a batch, optionally followed by standardise + clamp
 * (rcn.rs:407-412 / 86-89) with the model's scale_set. images: B images of H x W in `pixel_format`;
 * out: L x B. */
int rcn_cuda_features(rcn_cuda_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                      int standardise, double* out);
/* gen_scales (rcn.rs:230-251): mean and population sd over all L*B values; also stored as scale_set. */
int rcn_cuda_gen_scales(rcn_cuda_handle h, const double* feats, size_t L, size_t B, double* mean, double* sd);
/* v <- max((v-mean)/sd, 0) in place (rcn.rs:407-412). */
int rcn_cuda_standardise(rcn_cuda_handle h, double* feats, size_t n);

/* ---- inference: classify_test (rcn.rs:105-116), classify (rcn.rs:82-98), epoch eval (rcn.rs:152-157) */
int rcn_cuda_forward(rcn_cuda_handle h, const double* feats, size_t B, double* out_acts /* classes x B */);
/* argmax with last-max-wins (rcn.rs:92-97) of the forward pass. */
int rcn_cuda_classify_features(rcn_cuda_handle h, const double* feats, size_t B, int64_t* labels_out);
int rcn_cuda_classify(rcn_cuda_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                      int64_t* labels_out);
/* Number of samples whose {i : a_i == max a} equals {label} exactly (rcn.rs:153-157). */
int rcn_cuda_evaluate(rcn_cuda_handle h, const double* feats, const int64_t* labels, size_t B, uint64_t* accept);
/* Test-set evaluation (rcn.rs:152-157) straight from images: features + standardise with scale_set
 * (rcn.rs:84-89), forward, and per batch the quadratic cost sum_b 0.5*|a_L - y|^2 and the hit count of
 * rcn_cuda_evaluate. labels_out (optional, may be NULL) receives the rcn.rs:92-97 argmax of every sample.
 * images / labels / outputs may be host or device pointers. When images, labels, cost_out, accept_out and (if
 * given) labels_out are all in device memory the call does not synchronise; it can then be captured into a CUDA
 * graph once a call with at least as many images has run outside the capture (that call sizes the scratch
 * buffers, see rcn_cuda_allocation_generation). A host pointer among them makes the call synchronise.
 * Networks without the fused inference kernel (f64 pixels, a layer wider than 32, more than 4 layers) keep
 * features and activations of the whole batch in the model's grow-only scratch buffers after the call.
 * Leaves the gradient buffer, the epoch state and rcn_cuda_last_batch_stats untouched. */
int rcn_cuda_evaluate_images(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                             size_t B, size_t H, size_t W, double* cost_out, uint64_t* accept_out,
                             int64_t* labels_out);

/* ---- training: backprop (rcn.rs:260-314) + train_batch (rcn.rs:176-223) ------------------------ */
/* Targets: exactly one of `onehot` (classes x B, the reference's `y`) and `labels` (class index per sample,
 * expanded as get_expected_vec does, rcn.rs:466-471) must be non-NULL. */

/* Sum over the batch of backprop()'s (del_w, del_b), written to the model's flat gradient buffer
 * [dW0|db0|dW1|db1|...] -- the reduction of rcn.rs:190-205 without the update. */
int rcn_cuda_accumulate_gradients(rcn_cuda_handle h, const double* feats, const double* onehot,
                                  const int64_t* labels, size_t B);
/* Same, starting from raw images (features + standardise fused in front). */
int rcn_cuda_accumulate_gradients_images(rcn_cuda_handle h, const void* images, int pixel_format,
                                         const int64_t* labels, size_t B, size_t H, size_t W);
/* W <- W - (eta / batch) * sum_dW, b likewise (rcn.rs:210-222). `batch` is the GLOBAL minibatch size
 * (the data-parallel trainer all-reduces the gradient buffer between accumulate and apply). */
int rcn_cuda_apply_gradients(rcn_cuda_handle h, double eta, size_t batch);
/* train_batch (rcn.rs:176-223) = accumulate + apply on one device. */
int rcn_cuda_train_batch(rcn_cuda_handle h, const double* feats, const double* onehot, const int64_t* labels,
                         size_t B, double eta);
int rcn_cuda_train_batch_images(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                                size_t B, size_t H, size_t W, double eta);
/* Optional per-batch metric of the last accumulate/train call, evaluated with the PRE-update parameters:
 * quadratic cost sum_b 0.5*|a_L - y|^2 and the rcn.rs:153-157 hit count. */
int rcn_cuda_last_batch_stats(rcn_cuda_handle h, double* cost, uint64_t* hits);

/* ---- epoch mode: the inner loop of RCN::train (rcn.rs:144-149) over a dataset resident in HBM ------------
 * `for batch in training_set.chunks_exact(batch_size) { train_batch(batch, eta) }` with the batch selection done on
 * the DEVICE: step k trains on samples perm[pos .. pos+B) (perm == NULL: identity), pos advances by B after each
 * update and wraps to 0 once fewer than B samples remain (the remainder is dropped like chunks_exact does).
 * Nothing about a step depends on host state, so one captured CUDA graph replays for every step of every epoch
 * (re-shuffle by rewriting `perm` in place between epochs). All pointers must be DEVICE pointers and stay valid. */
int rcn_cuda_epoch_bind(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                        const int64_t* perm, size_t n_samples, size_t H, size_t W, size_t B);
int rcn_cuda_epoch_seek(rcn_cuda_handle h, size_t position);
int rcn_cuda_epoch_position(rcn_cuda_handle h, size_t* position); /* synchronises the stream */
/* accumulate: gradient sums of the current chunk into the gradient buffer; apply: update + advance. */
int rcn_cuda_epoch_accumulate(rcn_cuda_handle h);
int rcn_cuda_epoch_apply(rcn_cuda_handle h, double eta, size_t global_batch);
int rcn_cuda_epoch_step(rcn_cuda_handle h, double eta); /* accumulate + apply with global_batch = B */
/* n_steps consecutive epoch steps (rcn.rs:147-149: n_steps iterations of the chunks_exact loop) in one call. */
int rcn_cuda_epoch_run(rcn_cuda_handle h, double eta, size_t n_steps);

/* The same loop over a HOST-resident (already shuffled) dataset: `for batch in training_set.chunks_exact(B) {
 * train_batch(batch, eta) }` (rcn.rs:147-149). The host->device transfer of chunk k+1 overlaps the kernels of chunk k:
 * with PINNED u8 images and a narrow network the copy engine streams the chunks into a device ring ahead of the steps
 * (the first step starts after one chunk; the training kernel waits on an arrival counter in device memory), the steps
 * are replayed as CUDA graphs of up to 40 steps, and the step's result is written straight into pinned host memory;
 * otherwise double-buffered cudaMemcpyAsync on a copy stream. Every step's
 * result -- quadratic cost and rcn.rs:153-157 hit count under the pre-update parameters -- lands in cost_out / hits_out
 * (n_samples / B entries each, may be NULL). global_batch = 0 means B x (data-parallel world).
 * In a connected data-parallel group every rank calls this with its own shard of each global minibatch. */
int rcn_cuda_train_epoch_host(rcn_cuda_handle h, const void* images, int pixel_format, const int64_t* labels,
                              size_t n_samples, size_t H, size_t W, size_t B, double eta, size_t global_batch,
                              double* cost_out, uint64_t* hits_out, size_t* n_steps_out);

/* ---- data-parallel group: gradient exchange fused with the update over NVLink peer memory -------------------------
 * The reduction of rcn.rs:190-205 across the GPUs of one box (SURVEY.md 8e). After a group is connected,
 * rcn_cuda_apply_gradients / rcn_cuda_epoch_apply / rcn_cuda_train_epoch_host run ONE kernel that pushes this rank's
 * gradient sums into every peer's receive slots over NVLink, waits for the peers' pushes, adds the ranks in rank
 * order (replicas stay bit-identical) and applies W -= (eta / global_batch) * sum. No host-side collective call is
 * needed between accumulate and apply. Intended for latency-bound gradient sizes (up to ~1M parameters); larger
 * models use an NCCL all-reduce on the bound gradient buffer instead (mercer_research_b200/trainer.py).
 *   dp_init          allocates this rank's communication block; ipc_handle_out (64 bytes, may be NULL) receives its
 *                    cudaIpcMemHandle_t for ranks living in other processes.
 *   dp_connect_ipc   all_handles = world x 64 bytes, the handles of ranks 0..world-1 (own entry ignored).
 *   dp_connect_local group = world handles living in THIS process (one per device; peer access is enabled).
 * Every rank must execute the same sequence of apply calls, and in a connected group every accumulate must be followed by
 * exactly one apply before the next accumulate (the fused small-network kernels already push their gradients to the peers
 * at the end of accumulate, so that the exchange overlaps the launch of the update).
 * A receive never waits forever: a peer that stays silent for RCN_CUDA_DP_TIMEOUT_MS (default 10 000) sets a sticky error
 * word in this rank's block, the affected sums become NaN, and rcn_cuda_dp_error (which synchronises the stream) returns
 * RCN_ERR_STATE with *error = 1 -- the reference's equivalent is a poisoned mutex panic (rcn.rs:192-193). */
int rcn_cuda_dp_init(rcn_cuda_handle h, int world, int rank, void* ipc_handle_out);
int rcn_cuda_dp_connect_ipc(rcn_cuda_handle h, const void* all_handles);
int rcn_cuda_dp_connect_local(rcn_cuda_handle h, const rcn_cuda_handle* group);
int rcn_cuda_dp_shutdown(rcn_cuda_handle h);
int rcn_cuda_dp_error(rcn_cuda_handle h, int* error);

/* Device-side launch timeline of the fused step kernels (kernel 0 = forward/backward kernel A, 1 = weight-gradient kernel
 * B, 2 = data-parallel exchange kernel): per launch the earliest CTA start and the latest CTA end in %globaltimer
 * nanoseconds, kept for the last 64 launches -- the durations of, and gaps between, the kernels of a REPLAYED CUDA graph.
 * enable(1) allocates and clears the block (steps captured before the call must be re-captured: the allocation generation
 * is bumped); read: stamps = [2][4][64] uint64 (starts, then ends; slot = launch index % 64), launches = [4] uint32. */
int rcn_cuda_timeline_enable(rcn_cuda_handle h, int on);
int rcn_cuda_timeline_read(rcn_cuda_handle h, uint64_t* stamps, uint32_t* launches);

/* Gradient buffer access for the data-parallel trainer. bind: use caller-owned DEVICE memory (e.g. a torch
 * tensor that NCCL all-reduces) as the flat gradient buffer; NULL restores the internal one. */
int rcn_cuda_bind_gradient_buffer(rcn_cuda_handle h, double* device_ptr, size_t n);
int rcn_cuda_gradient_buffer(rcn_cuda_handle h, double** device_ptr, size_t* n);
int rcn_cuda_get_gradients(rcn_cuda_handle h, double* flat, size_t n);
/* Debug / parity taps of the last accumulate call: activations a_l (rows_l x B) and deltas (rows_l x B). */
int rcn_cuda_get_activations(rcn_cuda_handle h, size_t layer, double* out);
int rcn_cuda_get_deltas(rcn_cuda_handle h, size_t layer, double* out);

/* ---- launch accounting (bench.py: gpu_launches, per-kernel durations for the roofline) ------------------ */
/* Number of kernels this library has launched in this process. */
int rcn_cuda_kernel_launches(uint64_t* count);
/* Generation of the library's grow-only device buffers: changes whenever one of them is (re)allocated, i.e. whenever a
 * call needed more scratch than any call before it.  A caller that has captured library calls into its own CUDA graph
 * (device pointers baked in) compares the value from capture time before each replay and re-captures on a change; the
 * library's own step graphs (rcn_cuda_train_epoch_host) do the same internally.  scale_set is the other thing a captured
 * step holds BY VALUE (kernel arguments): re-capture after rcn_cuda_set_scale / rcn_cuda_gen_scales changed it. */
int rcn_cuda_allocation_generation(uint64_t* generation);
/* on != 0: start bracketing every kernel launch with CUDA events on its stream (clears old records);
 * on == 0: stop.  Adds two event records per launch -- never enable inside a timed region. */
int rcn_cuda_profile_enable(int on);
/* Synchronises the device and writes a JSON object {"kernel": {"launches": n, "total_ms": t}, ...} for the
 * records collected since the last enable. */
int rcn_cuda_profile_report(char* json_out, size_t capacity);

/* ---- op-level API: traits Convolve2D (kernel.rs:61-100) and Pool2D (kernel.rs:219-236) -------- */
/* These need no model; `device` selects the GPU and `cuda_stream` may be NULL. Outputs are caller-allocated:
 * convolve_2d: H x W (Same) or (H-kh+1) x (W-kw+1) (None); pool_2d: ceil(H/2) x ceil(W/2) (Same) or
 * floor (None). */
int rcn_cuda_convolve_2d(int device, void* cuda_stream, const double* m, size_t H, size_t W, const double* kernel,
                         size_t kh, size_t kw, int padding, double* out);
int rcn_cuda_convolve_2d_separated(int device, void* cuda_stream, const double* m, size_t H, size_t W, int op,
                                   int padding, double* out);
int rcn_cuda_relu(int device, void* cuda_stream, const double* m, size_t n, double* out);
/* argmax_out (optional, may be NULL) is this library's extension: index 2*dy+dx of the chosen element with
 * the reference's last-maximal-element-wins rule (kernel.rs:273-281). */
int rcn_cuda_pool_2d(int device, void* cuda_stream, const double* m, size_t H, size_t W, int padding, int pooling,
                     double* out, uint8_t* argmax_out);

/* ---- EXTENSIONS: operations BASELINE.json's north_star names that the reference does NOT implement ---------------
 * (SURVEY.md section 8a rows x1-x3; "parity unpinned": no reference code, test or golden vector exists, the checker
 * is oracle/ext_oracle.cpp written from the definitions.)  Conventions extend the reference's own: cross-correlation
 * without kernel flip and Padding::{None,Same} as Convolve2D::convolve_2d (kernel.rs:110-194); the 2x2 / stride-2
 * window, bottom/right zero padding and last-maximal-element rule of Pool2D::pool_2d (kernel.rs:245-349).
 * Tensors with channels are NHWC f64: x[((b*H + y)*W + x)*C + c]; weights w[co][ky][kx][ci]; dense-head matrices stay
 * column-major (n x B).  `device` / `cuda_stream` / host-or-device pointers as for the op-level API above. */
enum { RCN_ACT_NONE = 0, RCN_ACT_RELU = 1, RCN_ACT_SIGMOID = 2 };

/* x1: learned convolution.  y = act(conv(x, w) + bias); Same keeps H x W (odd kernels), None gives (H-kh+1) x (W-kw+1). */
int rcn_cuda_ext_conv2d_forward(int device, void* cuda_stream, const double* x, size_t B, size_t H, size_t W, size_t Ci,
                                const double* w, const double* bias /* may be NULL */, size_t Co, size_t kh, size_t kw,
                                int padding, int activation, double* y);
/* dz = dy .* act'(y), with act' expressed through the stored output y (sigmoid: y(1-y), relu: y > 0). */
int rcn_cuda_ext_activation_backward(int device, void* cuda_stream, const double* y, const double* dy, size_t n,
                                     int activation, double* dz);
/* dx = conv_transpose(dz, w), optionally fused with the previous layer's activation derivative:
 * dx .*= act_prev'(y_prev) when y_prev != NULL (y_prev has x's shape).  H, W, Ci describe x. */
int rcn_cuda_ext_conv2d_backward_data(int device, void* cuda_stream, const double* dz, size_t B, size_t H, size_t W,
                                      size_t Ci, const double* w, size_t Co, size_t kh, size_t kw, int padding,
                                      const double* y_prev, int activation_prev, double* dx);
/* dw[co][ky][kx][ci] = sum over batch and pixels of dz * x (deterministic fixed-order split reduction); db[co] = sum dz
 * (db may be NULL). */
int rcn_cuda_ext_conv2d_backward_weight(int device, void* cuda_stream, const double* x, const double* dz, size_t B, size_t H,
                                        size_t W, size_t Ci, size_t Co, size_t kh, size_t kw, int padding, double* dw,
                                        double* db);
/* x2: NHWC pooling, 2x2 window / stride 2.  pooling = RCN_POOLING_MAX or RCN_POOLING_AVERAGE (divides by 4 always).
 * argmax_out (max only, may be NULL): 2*dy+dx of the chosen element, last maximal element wins. */
int rcn_cuda_ext_pool2d_forward(int device, void* cuda_stream, const double* x, size_t B, size_t H, size_t W, size_t C,
                                int padding, int pooling, double* y, uint8_t* argmax_out);
/* H, W describe the pooling INPUT; dy / argmax have the pooled shape.  Max: dy is routed to the argmax element
 * (dropped when that element is the zero padding); average: dy / 4 to every in-bounds element of the window. */
int rcn_cuda_ext_pool2d_backward(int device, void* cuda_stream, const double* dy, const uint8_t* argmax, size_t B, size_t H,
                                 size_t W, size_t C, int padding, int pooling, double* dx);
/* x3: softmax + cross-entropy on column-major logits z (n x B): probs = softmax(z_b), loss[b] = -sum_i y_i log p_i,
 * delta = probs - y (gradient of loss[b] w.r.t. z_b).  Exactly one of onehot (n x B) / labels (B); any output may be NULL. */
int rcn_cuda_ext_softmax_xent(int device, void* cuda_stream, const double* z, size_t n, size_t B, const double* onehot,
                              const int64_t* labels, double* probs, double* loss, double* delta);

/* The GEMM building block of the dense and convolution layers, exposed for testing and benchmarking:
 * C (M x N, column-major) = A * B with A(m,k) = a_kcontig ? A[m*lda + k] : A[k*lda + m] and
 * B(k,n) = b_kcontig ? B[n*ldb + k] : B[k*ldb + n].
 *   impl 0: f64 tensor path (DMMA, mma.sync.m8n8k4.f64), cp.async-staged.
 *   impl 1: tcgen05 / TMEM / TMA integer-slice path: both operands are written as five balanced base-256 digit planes
 *           (int8) under per-row power-of-two scales, the 15 plane products with i+j <= 4 run as exact s8 x s8 -> s32
 *           tensor-core MMAs and are recombined in f64 (truncation ~ 6e-11 of the result; operands must be finite;
 *           K <= 16384).
 * The dense layers pick impl 1 automatically for large shapes (env RCN_CUDA_GEMM = dmma | tc | simt overrides). */
int rcn_cuda_ext_gemm_f64(int device, void* cuda_stream, const double* A, size_t lda, int a_kcontig, const double* B,
                          size_t ldb, int b_kcontig, size_t M, size_t N, size_t K, int impl, double* C);

/* ---- convolutional network: learned conv / pool layers in front of the dense stack ---------------------------------
 * EXTENSION (BASELINE.json north_star configs 3 and 4; the reference has no learned convolution).  The network is
 *   input (B, H, W, C)  ->  conv / pool stack (NHWC)  ->  flatten  ->  the reference's dense stack (sigmoid layers,
 *   quadratic cost, W -= (eta/B) * sum dW), or with RCN_HEAD_SOFTMAX_XENT the same stack with a softmax cross-entropy head.
 * layer_spec: n_layers records of RCN_CNN_LAYER_INTS int32 each:
 *   {RCN_CNN_CONV, Co, kh, kw, padding}   learned cross-correlation with bias, ALWAYS followed by ReLU; conventions and
 *                                         contract errors of rcn_cuda_ext_conv2d_forward (odd kernels for Same)
 *   {RCN_CNN_POOL, pooling, padding, 0, 0} 2x2 / stride 2 as rcn_cuda_ext_pool2d_forward (last maximal element wins, Same
 *                                         pads the bottom row / right column)
 * Flatten: the last stack output [B][Hp][Wp][C] IS the L x B column-major feature matrix of the dense stack,
 * L = Hp*Wp*C (sample-major NHWC order).  The dense stack is feedforward[0..n_ff) then `classes`; its features are NOT
 * standardised.
 * Parameters and gradients are one flat buffer [w0 (Co,kh,kw,Ci) | b0 (Co) | w1 | b1 | ... | W0 | b0 | W1 | b1 | ...]: the
 * conv layers in stack order, then the dense layers in the layout of rcn_cuda_set_params.
 * Images: RCN_PIXELS_U8_ROWMAJOR (B, H, W) with in_channels == 1, or RCN_PIXELS_F64_NHWC (B, H, W, in_channels); the shape
 * is fixed at creation (it fixes L and so the parameter count): other H, W fail with RCN_ERR_SHAPE.
 * Pointers may be host or device memory as elsewhere; with device images, labels and outputs nothing synchronises, and
 * once a call with at least as many images has sized the buffers (rcn_cuda_allocation_generation), accumulate + apply can
 * be captured into a CUDA graph.  A NaN reaching a max pool is not reported (the cost turns NaN instead).
 * Epoch mode (rcn_cuda_cnn_epoch_*, below) trains over a dataset resident in device memory with a device-side cursor, like
 * rcn_cuda_epoch_*; each step gathers its images and labels with one staging kernel. */
enum { RCN_CNN_CONV = 0, RCN_CNN_POOL = 1 };
#define RCN_CNN_LAYER_INTS 5
/* Output head of the network's dense stack.
 *   RCN_HEAD_SIGMOID_QUADRATIC  the reference's: sigmoid output layer, cost sum_b 0.5 |a_b - y_b|^2, delta_L = (a - y) a (1 - a),
 *                               a hit when {i : a_i = max a} = {label} (rcn.rs:153-157), labels the last-max-wins argmax of a.
 *   RCN_HEAD_SOFTMAX_XENT       hidden layers unchanged (sigmoid, delta_l = (W_{l+1}^T delta_{l+1}) a (1 - a)); the output
 *                               layer is affine, z = W a + b, and p = softmax(z) per sample with rcn_cuda_ext_softmax_xent's
 *                               arithmetic (m = max z, then s = sum exp(z - m), then log s).  Cost per sample
 *                               (log s + m) - z_label, summed over the batch; delta_L = p - onehot(label).  Hits and labels
 *                               are decided on z, not on p (exp rounding can make distinct logits equal probabilities): a hit
 *                               when {i : z_i = max z} = {label}, labels the last-max-wins argmax of z.  A label outside
 *                               [0, classes) has an all-zero target (cost 0, delta = p); a non-finite logit makes that
 *                               sample's p, delta and cost NaN.
 * Both heads update with W -= (eta / B) * sum dW. */
enum { RCN_HEAD_SIGMOID_QUADRATIC = 0, RCN_HEAD_SOFTMAX_XENT = 1 };
/* Validates the whole spec before any device work (status codes and messages of the ext ops; a zero-width dense layer or
 * zero classes is RCN_ERR_INVALID).  Parameters start at zero: set them with rcn_cuda_cnn_set_params.
 * rcn_cuda_cnn_create is rcn_cuda_cnn_create_with_head with RCN_HEAD_SIGMOID_QUADRATIC; an unknown head is RCN_ERR_INVALID. */
int rcn_cuda_cnn_create(int device, size_t H, size_t W, size_t in_channels, const int32_t* layer_spec, size_t n_layers,
                        const size_t* feedforward, size_t n_ff, size_t classes, rcn_cuda_cnn_handle* out);
int rcn_cuda_cnn_create_with_head(int device, size_t H, size_t W, size_t in_channels, const int32_t* layer_spec, size_t n_layers,
                                  const size_t* feedforward, size_t n_ff, size_t classes, int head, rcn_cuda_cnn_handle* out);
int rcn_cuda_cnn_destroy(rcn_cuda_cnn_handle h);
/* As rcn_cuda_set_stream: NULL is the legacy default stream, RCN_STREAM_OWN the handle's own stream. */
int rcn_cuda_cnn_set_stream(rcn_cuda_cnn_handle h, void* cuda_stream);
int rcn_cuda_cnn_synchronize(rcn_cuda_cnn_handle h);
/* Output shape of stack layer `layer` (n_layers - 1: the flattened features, L = H*W*C). */
int rcn_cuda_cnn_layer_shape(rcn_cuda_cnn_handle h, size_t layer, size_t* H, size_t* W, size_t* C);
int rcn_cuda_cnn_param_count(rcn_cuda_cnn_handle h, size_t* n);
int rcn_cuda_cnn_set_params(rcn_cuda_cnn_handle h, const double* flat, size_t n);
int rcn_cuda_cnn_get_params(rcn_cuda_cnn_handle h, double* flat, size_t n);
/* Gradient sums of the batch into the flat gradient buffer, no update.  Per step: conv (+bias+ReLU) and pool forward, the
 * dense stack's accumulate on the stack output, dX = W0^T delta0 with the pre-update W0, then down the stack pool
 * backward, ReLU', conv weight and bias gradients, and conv input gradients except for the first conv layer. */
int rcn_cuda_cnn_accumulate(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                            size_t H, size_t W);
/* p <- p - (eta / global_batch) * g over every parameter (rcn.rs:210-222 rounding), or the step of the optimizer set with
 * rcn_cuda_cnn_set_optimizer (below). */
int rcn_cuda_cnn_apply(rcn_cuda_cnn_handle h, double eta, size_t global_batch);
/* accumulate + apply(eta, B) */
int rcn_cuda_cnn_train_batch(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                             size_t H, size_t W, double eta);
/* The head's cost and the head's hit count (rule above) of the last accumulate, under the pre-update parameters. */
int rcn_cuda_cnn_last_batch_stats(rcn_cuda_cnn_handle h, double* cost, uint64_t* hits);
/* Epoch mode: `for batch in training_set.chunks_exact(B) { train_batch(batch, eta) }` (rcn.rs:144-149) over a dataset in
 * DEVICE memory, with meaning, contract and status codes of rcn_cuda_epoch_*: step k trains on samples perm[pos .. pos+B)
 * (perm == NULL: identity); pos advances by B with each apply and wraps to 0 once fewer than B samples remain.
 *   bind        images (n_samples images in `pixel_format`, H x W as the network was created for: RCN_ERR_SHAPE otherwise),
 *               labels (n_samples) and perm (n_samples, may be NULL) must be device pointers (RCN_ERR_INVALID otherwise)
 *               and stay valid while bound; n_samples >= B > 0 (RCN_ERR_INVALID).  Every entry of perm must lie in
 *               [0, n_samples): the caller's contract, not checked.  Reserves the step's buffers for B, sets the cursor
 *               to 0 and drains the stream.  perm may be rewritten in place between steps (re-shuffle per epoch).
 *   accumulate  one kernel gathers chunk perm[pos .. pos+B) and its labels (u8 images: with the f64 copy the first layer's
 *               weight gradient reads), then rcn_cuda_cnn_accumulate's work on it; the cursor does not move, so two
 *               accumulates without an apply see the same chunk.
 *   apply       rcn_cuda_cnn_apply, and the cursor advances.
 * Every step entry point before a bind fails with RCN_ERR_STATE.  After bind and one accumulate outside a capture a step
 * neither allocates nor synchronises, so one captured step replays for every step of every epoch; re-capture when
 * rcn_cuda_allocation_generation changed.  The layer buffers are shared with evaluate / classify: those calls on more than
 * B images grow them (and move them), which a captured step notices only through that generation. */
int rcn_cuda_cnn_epoch_bind(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels,
                            const int64_t* perm, size_t n_samples, size_t H, size_t W, size_t B);
int rcn_cuda_cnn_epoch_seek(rcn_cuda_cnn_handle h, size_t position);
int rcn_cuda_cnn_epoch_position(rcn_cuda_cnn_handle h, size_t* position); /* synchronises the stream */
int rcn_cuda_cnn_epoch_accumulate(rcn_cuda_cnn_handle h);
int rcn_cuda_cnn_epoch_apply(rcn_cuda_cnn_handle h, double eta, size_t global_batch);
int rcn_cuda_cnn_epoch_step(rcn_cuda_cnn_handle h, double eta); /* accumulate + apply with global_batch = B */
int rcn_cuda_cnn_epoch_run(rcn_cuda_cnn_handle h, double eta, size_t n_steps); /* n_steps epoch steps in one call */
/* Forward pass only: cost_out the head's batch cost, accept_out the count of hits under the head's hit rule, labels_out
 * (optional) the head's labels (the rcn.rs:92-97 last-max-wins argmax, of z with the softmax head).
 * Leaves the gradients and the last-batch statistics untouched (the layer-output tap then shows this batch). */
int rcn_cuda_cnn_evaluate_images(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                                 size_t H, size_t W, double* cost_out, uint64_t* accept_out, int64_t* labels_out);
/* The head's labels of B images, as evaluate's labels_out. */
int rcn_cuda_cnn_classify_images(rcn_cuda_cnn_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                                 int64_t* labels_out);
/* As rcn_cuda_bind_gradient_buffer / rcn_cuda_gradient_buffer / rcn_cuda_get_gradients, over the whole flat buffer. */
int rcn_cuda_cnn_bind_gradient_buffer(rcn_cuda_cnn_handle h, double* device_ptr, size_t n);
int rcn_cuda_cnn_gradient_buffer(rcn_cuda_cnn_handle h, double** device_ptr, size_t* n);
int rcn_cuda_cnn_get_gradients(rcn_cuda_cnn_handle h, double* flat, size_t n);
/* Debug / parity taps: the output of stack layer `layer` of the last accumulate or evaluate (post-ReLU for a conv, pooled
 * for a pool; B x H x W x C), and the dense stack's input gradient dX (L x B) of the last accumulate. */
int rcn_cuda_cnn_get_layer_output(rcn_cuda_cnn_handle h, size_t layer, double* out);
int rcn_cuda_cnn_get_input_gradient(rcn_cuda_cnn_handle h, double* out);
/* Optimizer of the network's apply / epoch_apply (the update above is the default; RCN has no optimizer choice).
 * Let g be a parameter's gradient sum (the flat buffer, after any all-reduce), B the global batch, eta the learning rate
 * and lambda the weight decay, which applies to every parameter.  Every product, sum, quotient and square root is rounded
 * on its own (no fused multiply-add), in this order:
 *   RCN_OPTIMIZER_SGD     momentum mu in [0, 1), nesterov 0 / 1 (needs mu > 0), weight_decay lambda >= 0.  The default.
 *                         mu = lambda = 0 is the plain update W -= (eta / B) * g, unchanged.  Otherwise (torch.optim.SGD
 *                         without dampening; v starts at 0):
 *                           gh = g / B;  d = gh + lambda * p;  v = mu * v + d;  u = nesterov ? d + mu * v : v;  p = p - eta * u
 *                         (with mu = 0 there is no v and u = d).
 *   RCN_OPTIMIZER_ADAMW   beta1, beta2 in [0, 1), eps > 0, weight_decay lambda >= 0 (torch.optim.AdamW).  The device keeps
 *                         t and the running products beta1^t, beta2^t (from 0, 1, 1).  Per step t += 1, b1 = beta1^t * beta1,
 *                         b2 = beta2^t * beta2 (stored back as the new beta1^t, beta2^t), then per parameter
 *                           p = p * (1 - eta * lambda)            (the factor formed once on the host)
 *                           gh = g / B;  m = beta1 * m + (1 - beta1) * gh;  v = beta2 * v + (1 - beta2) * (gh * gh)
 *                           p = p - eta * ((m / (1 - b1)) / (sqrt(v / (1 - b2)) + eps))
 * apply with global_batch 0 changes nothing, t included.  set_optimizer checks the hyperparameters of `kind` (those of the
 * other kind are ignored; an unknown kind, a value out of range or a non-finite one is RCN_ERR_INVALID before any device
 * work), allocates and resets the state and bumps rcn_cuda_allocation_generation, so a captured step must be re-captured
 * (it also holds eta and the hyperparameters by value).  A step itself never allocates.
 * The state is a flat f64 vector with the layout of the gradient buffer: v (n_params) for SGD with mu > 0, m | v | t,
 * beta1^t, beta2^t (2 n_params + 3) for AdamW, empty otherwise.  get / set copy it (n must be the state size:
 * RCN_ERR_INVALID otherwise); set moves no buffer, so the allocation generation stays. */
enum { RCN_OPTIMIZER_SGD = 0, RCN_OPTIMIZER_ADAMW = 1 };
int rcn_cuda_cnn_set_optimizer(rcn_cuda_cnn_handle h, int kind, double momentum, int nesterov, double weight_decay, double beta1,
                               double beta2, double eps);
int rcn_cuda_cnn_optimizer_state_size(rcn_cuda_cnn_handle h, size_t* n);
int rcn_cuda_cnn_get_optimizer_state(rcn_cuda_cnn_handle h, double* state, size_t n);
int rcn_cuda_cnn_set_optimizer_state(rcn_cuda_cnn_handle h, const double* state, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* RCN_CUDA_H */
