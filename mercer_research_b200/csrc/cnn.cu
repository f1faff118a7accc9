// cnn.cu -- EXTENSION (not in the reference): a trainable network of learned convolution and pooling layers in front of
// the reference's dense stack (BASELINE.json north_star configs 3 and 4; SURVEY.md section 8a rows x1, x2).
//
//   images -> [conv (+bias, ReLU) | pool]* -> flatten -> dense stack (sigmoid, quadratic cost) -> SGD on every parameter
//
// (or momentum SGD / AdamW, rcn_cuda_cnn_set_optimizer: one optim.cu launch over the conv and the dense parameters)
//
// or, created with RCN_HEAD_SOFTMAX_XENT, the same dense stack with an affine output layer, softmax and cross-entropy
// (semantics in rcn_cuda.h).  The head lives in the dense model (model_set_head): its last layer stores the logits and
// softmax_xent_head_kernel turns them into p, delta_L = p - y and the batch statistics; the backward pass below is the same
// for both heads.
//
// The handle owns the conv parameters, the per-layer activations and a dense rcn_cuda_model (model.cu) created with an
// empty convpool stack, whose gradient buffer is the tail of this handle's flat gradient buffer.  A step only launches
// kernels that already exist as ops (conv.cu, extops.cu, dense.cu, smallnet.cu), plus the dense stack's input gradient
// (launch_dense_input_grad) and cnn_stage_batch_kernel: for u8 images the widening copy the first layer's weight gradient
// reads, and in epoch mode the gather of the step's images and labels from the bound dataset (that copy included):
//   forward    per conv layer  conv2d forward, bias + ReLU in its epilogue (direct kernel / DMMA / tcgen05 implicit GEMM)
//              per pool layer  ext_pool_forward_kernel (argmax bytes kept for the backward pass)
//              dense stack     the model's accumulate on the last output (fused kernels A/B on narrow heads), delta0 kept
//   backward   dX = W0^T delta0 (pre-update W0), then down the stack: pool backward; ReLU' (activation_backward, or fused
//              into the conv backward-data epilogue when the layer below is a conv); conv weight + bias gradients straight
//              into the flat buffer; conv backward-data unless no conv layer lies below.
// Flatten needs no kernel: the last output [B][Hp][Wp][C] is the L x B column-major matrix the dense code reads.
#include <algorithm>
#include <memory>
#include <new>
#include <vector>

#include "cnn.cuh"
#include "conv.cuh"
#include "dense.cuh"
#include "optim.cuh"
#include "ozaki.cuh"

namespace rcn {

template <int VEC> struct StageVec;
template <> struct StageVec<16> { using T = uint4; };
template <> struct StageVec<8> { using T = uint2; };
template <> struct StageVec<4> { using T = unsigned; };
template <> struct StageVec<1> { using T = uint8_t; };

__device__ __forceinline__ unsigned stage_word(const uint4& v, int j) { return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w; }
__device__ __forceinline__ unsigned stage_word(const uint2& v, int j) { return j == 0 ? v.x : v.y; }
__device__ __forceinline__ unsigned stage_word(unsigned v, int) { return v; }

// Builds a step's input from a dataset in device memory: chunk image b is dataset image perm[c + b] (perm == NULL: c + b)
// with c = *cursor, read once (cursor == NULL: 0).  chunk (optional) receives the images as stored, x64 (optional, u8
// images) their f64 widening, labels_batch (optional) labels[perm[c + b]].  Each thread copies one VEC-byte vector
// (b, k) of the chunk per iteration, so every thread of the grid has a load in flight, whatever the image size; VEC
// divides img_bytes and the alignment of `images` and `chunk` (launch_stage_batch picks it), and for VEC >= 2 the widened
// copy goes out in 16-byte stores.  (b, k) advances by the grid stride without a division inside the loop.
template <int VEC>
__global__ void __launch_bounds__(256) cnn_stage_batch_kernel(const uint8_t* __restrict__ images, size_t img_bytes,
                                                              const int64_t* __restrict__ perm,
                                                              const long long* __restrict__ cursor, size_t B,
                                                              const int64_t* __restrict__ labels,
                                                              int64_t* __restrict__ labels_batch, uint8_t* __restrict__ chunk,
                                                              double* __restrict__ x64) {
    using V = typename StageVec<VEC>::T;
    const long long c = cursor ? __ldcg(cursor) : 0;   // the previous step's update wrote it
    const size_t nv = img_bytes / VEC;                 // vectors per image
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t sb = stride / nv, sk = stride - sb * nv;
    const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    size_t b = t / nv, k = t - b * nv;
    while (b < B) {
        const long long i = perm ? __ldg(perm + c + (long long)b) : c + (long long)b;
        if (labels_batch && k == 0) labels_batch[b] = __ldg(labels + i);
        const V v = __ldg(reinterpret_cast<const V*>(images + (size_t)i * img_bytes) + k);
        if (chunk) reinterpret_cast<V*>(chunk + b * img_bytes)[k] = v;
        if (x64) {
            double* wide = x64 + b * img_bytes + k * VEC;
            if constexpr (VEC == 1) {
                wide[0] = (double)v;
            } else {
                double2* w2 = reinterpret_cast<double2*>(wide);
#pragma unroll
                for (int j = 0; j < VEC; j += 2) {
                    const unsigned wd = stage_word(v, j >> 2);
                    const int s = (j & 3) * 8;
                    w2[j >> 1] = make_double2((double)((wd >> s) & 0xffu), (double)((wd >> (s + 8)) & 0xffu));
                }
            }
        }
        b += sb;
        k += sk;
        if (k >= nv) { k -= nv; ++b; }
    }
}

struct CnnLayer {
    int kind = RCN_CNN_CONV;
    int pooling = 0, padding = 0;
    size_t kh = 0, kw = 0;
    size_t Hi = 0, Wi = 0, Ci = 0, Ho = 0, Wo = 0, Co = 0;   // input and output maps (a pool keeps the channels)
    size_t w_off = 0, b_off = 0;                            // conv: offsets in the flat parameter buffer
    DevBuf out, argmax;
    size_t out_len() const { return Ho * Wo * Co; }
};

}  // namespace rcn

using namespace rcn;

struct rcn_cuda_cnn {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    size_t H = 0, W = 0, Cin = 0, L = 0;
    std::vector<CnnLayer> layers;
    size_t n_conv = 0, n_params = 0;   // conv parameters (head of the flat buffer), all parameters
    size_t max_len = 0;                // largest map of the stack, per sample (gradient scratch)
    rcn_cuda_model* dense = nullptr;
    DevBuf params, grads_own;          // params: the conv part; the dense part lives in the model
    double* grads = nullptr;
    DevBuf in_stage, lab_stage, out_stage, x64, dx, gbuf[2], flip_ws, wgrad_ws, small;
    ReduceScratch rs;
    OzakiWorkspace oz;
    size_t out_B = 0;                  // batch of the last forward (layer-output taps)
    size_t grad_B = 0;                 // batch of the last accumulate (input-gradient tap)
    // epoch mode: the bound dataset (caller's device memory), the staged chunk and the state block
    // ep_state = [cursor, padding, labels_batch[B]] (int64)
    const void* ep_images = nullptr;
    const int64_t* ep_labels = nullptr;
    const int64_t* ep_perm = nullptr;
    int ep_fmt = 0;
    size_t ep_n = 0, ep_B = 0;
    DevBuf ep_chunk, ep_state;
    // optimizer (rcn_cuda_cnn_set_optimizer): opt_state = [state (optim_state_len doubles) | AdamW's CTA ticket]
    OptimConfig opt;
    DevBuf opt_state;
};

namespace {

#define RCN_CNN_ENTER(h)                                                    \
    if (!(h)) return fail(RCN_ERR_INVALID, "null network handle");          \
    RCN_CUDA_TRY(cudaSetDevice((h)->device));

int deliver(rcn_cuda_cnn* h, void* dst, const void* dev_src, size_t bytes) {
    if (bytes == 0) return RCN_OK;
    if (is_device_ptr(dst)) {
        if (dst != dev_src) RCN_CUDA_TRY(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return RCN_OK;
    }
    RCN_CUDA_TRY(cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

// the geometry was validated at creation; the batch can still exceed the kernels' 32-bit pixel indices
int layer_shape(const CnnLayer& ly, size_t B, ConvShape* s) {
    return check_conv_shape(B, ly.Hi, ly.Wi, ly.Ci, ly.Co, ly.kh, ly.kw, ly.padding, s);
}

size_t image_bytes(const rcn_cuda_cnn* h, int fmt) { return h->H * h->W * h->Cin * (fmt == RCN_PIXELS_U8_ROWMAJOR ? 1 : 8); }

// The pixel format and the image size of a call against the network.
int check_images(const rcn_cuda_cnn* h, int fmt, size_t H, size_t W) {
    if (fmt != RCN_PIXELS_U8_ROWMAJOR && fmt != RCN_PIXELS_F64_NHWC)
        return fail(RCN_ERR_INVALID, "unknown pixel format %d (the network takes u8 row-major or f64 NHWC images)", fmt);
    if (fmt == RCN_PIXELS_U8_ROWMAJOR && h->Cin != 1)
        return fail(RCN_ERR_SHAPE, "u8 images have one channel, the network takes %zu", h->Cin);
    if (H != h->H || W != h->W)
        return fail(RCN_ERR_SHAPE, "the network was created for %zu x %zu images, got %zu x %zu", h->H, h->W, H, W);
    return RCN_OK;
}

// cnn_stage_batch_kernel over B images of img_bytes each; the widest access that img_bytes and both byte pointers allow.
int launch_stage_batch(rcn_cuda_cnn* h, const void* images, size_t img_bytes, const int64_t* perm, const long long* cursor,
                       size_t B, const int64_t* labels, int64_t* labels_batch, void* chunk, double* x64) {
    if (B == 0) return RCN_OK;
    const uintptr_t align = (uintptr_t)images | (uintptr_t)chunk;
    int vec = 1;
    for (int v : {16, 8, 4})
        if (img_bytes % v == 0 && align % v == 0) { vec = v; break; }
    // one vector per thread, grid-stride beyond 8 CTAs per SM
    const unsigned grid = (unsigned)std::min<size_t>((B * (img_bytes / vec) + 255) / 256, (size_t)kNumSMs * 8);
    const uint8_t* src = (const uint8_t*)images;
    uint8_t* dst = (uint8_t*)chunk;
#define RCN_STAGE_LAUNCH(V)                                                                                                  \
    RCN_LAUNCH("cnn_stage_batch_kernel", h->stream,                                                                          \
               cnn_stage_batch_kernel<V><<<grid, 256, 0, h->stream>>>(src, img_bytes, perm, cursor, B, labels, labels_batch, \
                                                                      dst, x64))
    switch (vec) {
        case 16: RCN_STAGE_LAUNCH(16); break;
        case 8: RCN_STAGE_LAUNCH(8); break;
        case 4: RCN_STAGE_LAUNCH(4); break;
        default: RCN_STAGE_LAUNCH(1); break;
    }
#undef RCN_STAGE_LAUNCH
    return RCN_OK;
}

// Checks the call's images against the network and stages them (and the labels, when given) on the handle's stream.
int stage_inputs(rcn_cuda_cnn* h, const void* images, int fmt, const int64_t* labels, size_t B, size_t H, size_t W,
                 const void** img_dev, const int64_t** lab_dev, bool* host_in) {
    RCN_TRY(check_images(h, fmt, H, W));
    if (!images) return fail(RCN_ERR_INVALID, "null images");
    StagedIn in;
    RCN_TRY(in.stage(images, B * image_bytes(h, fmt), h->in_stage, h->stream, host_in));
    *img_dev = in.dev;
    if (lab_dev) {
        if (!labels) return fail(RCN_ERR_INVALID, "null labels");
        StagedIn lb;
        RCN_TRY(lb.stage(labels, B * sizeof(int64_t), h->lab_stage, h->stream, host_in));
        *lab_dev = (const int64_t*)lb.dev;
    }
    return RCN_OK;
}

// The conv / pool stack on device images.  `training`: keep the max-pool argmax bytes and an f64 copy of u8 images for the
// first conv layer's weight gradient (`x64_staged`: the epoch staging kernel already wrote that copy into x64).  Returns
// the first layer's f64 input (NULL when u8 images were read directly).
int forward_stack(rcn_cuda_cnn* h, const void* img, int fmt, size_t B, bool training, bool x64_staged, const double** x0) {
    const bool u8 = fmt == RCN_PIXELS_U8_ROWMAJOR;
    const CnnLayer& first = h->layers[0];
    ConvShape s0{};
    if (first.kind == RCN_CNN_CONV) RCN_TRY(layer_shape(first, B, &s0));
    const bool direct_u8 = u8 && first.kind == RCN_CNN_CONV && conv_direct_ok(s0);
    const double* x = u8 ? nullptr : (const double*)img;
    if (u8 && (!direct_u8 || (training && first.kind == RCN_CNN_CONV))) {
        if (!x64_staged) {
            const size_t n = B * h->H * h->W;
            RCN_TRY(h->x64.reserve(n * sizeof(double)));
            RCN_TRY(launch_stage_batch(h, img, h->H * h->W, nullptr, nullptr, B, nullptr, nullptr, nullptr, h->x64.as<double>()));
        }
        x = h->x64.as<double>();
    }
    *x0 = x;
    int* nan_flag = reinterpret_cast<int*>(h->small.as<double>() + 4);
    const double* in = x;
    for (size_t l = 0; l < h->layers.size(); ++l) {
        CnnLayer& ly = h->layers[l];
        RCN_TRY(ly.out.reserve(B * ly.out_len() * sizeof(double)));
        double* y = ly.out.as<double>();
        if (ly.kind == RCN_CNN_CONV) {
            ConvShape s;
            RCN_TRY(layer_shape(ly, B, &s));
            const double* w = h->params.as<double>() + ly.w_off;
            const double* b = h->params.as<double>() + ly.b_off;
            if (l == 0 && direct_u8) RCN_TRY(launch_conv2d_forward_u8((const uint8_t*)img, w, b, s, ACT_RELU, y, h->stream));
            else RCN_TRY(launch_conv2d_forward(in, w, b, s, ACT_RELU, y, h->stream, &h->oz));
        } else {
            uint8_t* am = nullptr;
            if (training && ly.pooling == RCN_POOLING_MAX) {
                RCN_TRY(ly.argmax.reserve(B * ly.out_len()));
                am = ly.argmax.as<uint8_t>();
            }
            RCN_TRY(launch_pool2d_forward(in, B, ly.Hi, ly.Wi, ly.Ci, ly.Ho, ly.Wo, ly.pooling, y, am, nan_flag, h->stream));
        }
        in = y;
    }
    h->out_B = B;
    return RCN_OK;
}

int accumulate_dev(rcn_cuda_cnn* h, const void* img, int fmt, const int64_t* labels, size_t B, bool x64_staged = false) {
    if (B == 0) {
        RCN_CUDA_TRY(cudaMemsetAsync(h->grads, 0, h->n_params * sizeof(double), h->stream));
        return RCN_OK;
    }
    const double* x0 = nullptr;
    RCN_TRY(forward_stack(h, img, fmt, B, true, x64_staged, &x0));
    const size_t n = h->layers.size();
    RCN_TRY(rcn_cuda_accumulate_gradients(h->dense, h->layers[n - 1].out.as<double>(), nullptr, labels, B));
    // dX = W0^T delta0, read before apply moves W0
    const double *W0 = nullptr, *d0 = nullptr;
    size_t R0 = 0, L0 = 0;
    RCN_TRY(model_first_layer(h->dense, &W0, &d0, &R0, &L0));
    RCN_TRY(h->dx.reserve(h->L * B * sizeof(double)));
    RCN_TRY(launch_dense_input_grad(W0, d0, h->L, R0, B, h->dx.as<double>(), h->stream, &h->oz));
    h->grad_B = B;
    for (DevBuf& g : h->gbuf) RCN_TRY(g.reserve(B * h->max_len * sizeof(double)));
    // walk down the stack; g is the gradient with respect to layer l's output, already multiplied by ReLU' when g_is_dz;
    // gbuf[ping] never holds g
    const double* g = h->dx.as<double>();
    bool g_is_dz = false;
    int ping = 0;
    size_t first_conv = n;
    for (size_t l = 0; l < n; ++l)
        if (h->layers[l].kind == RCN_CNN_CONV) { first_conv = l; break; }
    for (size_t l = n; l-- > 0;) {
        const CnnLayer& ly = h->layers[l];
        const bool conv_below = first_conv < l;
        if (ly.kind == RCN_CNN_POOL) {
            if (!conv_below) break;
            double* gin = h->gbuf[ping].as<double>();
            ping ^= 1;
            RCN_TRY(launch_pool2d_backward(g, ly.argmax.as<uint8_t>(), B, ly.Hi, ly.Wi, ly.Ci, ly.Ho, ly.Wo, ly.pooling, gin,
                                           h->stream));
            g = gin;
            g_is_dz = false;
            continue;
        }
        ConvShape s;
        RCN_TRY(layer_shape(ly, B, &s));
        const double* dz = g;
        if (!g_is_dz) {
            double* t = h->gbuf[ping].as<double>();
            ping ^= 1;
            RCN_TRY(launch_activation_backward(ly.out.as<double>(), g, B * ly.out_len(), ACT_RELU, t, h->stream));
            dz = t;
        }
        const double* x_in = l == 0 ? x0 : h->layers[l - 1].out.as<double>();
        RCN_TRY(launch_conv2d_backward_weight(x_in, dz, s, h->grads + ly.w_off, h->grads + ly.b_off, h->wgrad_ws, h->stream, &h->oz,
                                              &h->rs));
        if (!conv_below) break;
        const bool fuse = h->layers[l - 1].kind == RCN_CNN_CONV;   // ReLU' of the conv below in the epilogue
        double* gin = h->gbuf[ping].as<double>();
        ping ^= 1;
        RCN_TRY(launch_conv2d_backward_data(dz, h->params.as<double>() + ly.w_off, s, fuse ? h->layers[l - 1].out.as<double>() : nullptr,
                                            fuse ? ACT_RELU : ACT_NONE, gin, h->flip_ws, h->stream, &h->oz));
        g = gin;
        g_is_dz = fuse;
    }
    return RCN_OK;
}

int accumulate(rcn_cuda_cnn* h, const void* images, int fmt, const int64_t* labels, size_t B, size_t H, size_t W) {
    if (B == 0) return accumulate_dev(h, nullptr, fmt, nullptr, 0);
    const void* img = nullptr;
    const int64_t* lab = nullptr;
    bool host_in = false;
    RCN_TRY(stage_inputs(h, images, fmt, labels, B, H, W, &img, &lab, &host_in));
    RCN_TRY(accumulate_dev(h, img, fmt, lab, B));
    if (host_in) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));   // the caller may reuse its host buffers
    return RCN_OK;
}

// The optimizer step of a non-default optimizer over the conv parameters and the dense model's, in one launch.
int optim_step(rcn_cuda_cnn* h, double eta, size_t batch, long long* cursor = nullptr) {
    double* dense = nullptr;
    size_t n_dense = 0;
    RCN_TRY(model_params(h->dense, &dense, &n_dense));
    double* st = h->opt_state.as<double>();
    unsigned* ticket = st ? reinterpret_cast<unsigned*>(st + optim_state_len(h->opt, h->n_params)) : nullptr;
    return launch_optim_update(h->opt, h->params.as<double>(), h->n_conv, dense, n_dense, h->grads, st, ticket, eta, batch,
                               h->stream, cursor, (long long)h->ep_B, (long long)h->ep_n);
}

int apply(rcn_cuda_cnn* h, double eta, size_t batch) {
    if (batch == 0) return RCN_OK;
    if (!optim_is_plain(h->opt)) return optim_step(h, eta, batch);
    // (eta / batch) formed first, then the rounded product subtracted (rcn.rs:214); the dense part forms the same scale
    if (h->n_conv) RCN_TRY(launch_sgd_update(h->params.as<double>(), h->grads, h->n_conv, eta / (double)batch, h->stream));
    return rcn_cuda_apply_gradients(h->dense, eta, batch);
}

// ---- epoch mode: rcn.rs:144-149 over a dataset resident in device memory ---------------------------------------------
constexpr size_t kCnnEpSlots = 2;   // ep_state: cursor, padding; labels_batch follows

int require_epoch(const rcn_cuda_cnn* h) {
    if (!h->ep_images) return fail(RCN_ERR_STATE, "no dataset bound: call rcn_cuda_cnn_epoch_bind first");
    return RCN_OK;
}

// Stages chunk perm[c .. c+B) (and for u8 images its f64 copy) and accumulates it; the cursor stays where it is.
int epoch_accumulate(rcn_cuda_cnn* h) {
    RCN_TRY(require_epoch(h));
    const bool u8 = h->ep_fmt == RCN_PIXELS_U8_ROWMAJOR;
    long long* st = h->ep_state.as<long long>();
    int64_t* lab = reinterpret_cast<int64_t*>(st + kCnnEpSlots);
    RCN_TRY(launch_stage_batch(h, h->ep_images, image_bytes(h, h->ep_fmt), h->ep_perm, st, h->ep_B, h->ep_labels, lab,
                               h->ep_chunk.p, u8 ? h->x64.as<double>() : nullptr));
    return accumulate_dev(h, h->ep_chunk.p, h->ep_fmt, lab, h->ep_B, u8);
}

// apply(), with the conv update also advancing the cursor by B (chunks_exact wrap-around, rcn.rs:147); with no conv
// parameters the update kernel runs on zero of them and only advances the cursor.
int epoch_apply(rcn_cuda_cnn* h, double eta, size_t batch) {
    RCN_TRY(require_epoch(h));
    if (batch == 0) return fail(RCN_ERR_INVALID, "global batch is zero");
    if (!optim_is_plain(h->opt)) return optim_step(h, eta, batch, h->ep_state.as<long long>());
    RCN_TRY(launch_sgd_update(h->params.as<double>(), h->grads, h->n_conv, eta / (double)batch, h->stream,
                              h->ep_state.as<long long>(), (long long)h->ep_B, (long long)h->ep_n));
    return rcn_cuda_apply_gradients(h->dense, eta, batch);
}

int copy_in(rcn_cuda_cnn* h, double* dst_dev, const double* src, size_t n) {
    if (n == 0) return RCN_OK;
    const bool dev = is_device_ptr(src);
    RCN_CUDA_TRY(cudaMemcpyAsync(dst_dev, src, n * sizeof(double), dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
    if (!dev) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

// Output maps of every layer and the parameter layout; every check the ext ops would make, before any device work.
int plan_layers(rcn_cuda_cnn* h, const int32_t* spec, size_t n_layers) {
    size_t Hc = h->H, Wc = h->W, Cc = h->Cin, off = 0;
    h->max_len = Hc * Wc * Cc;
    for (size_t l = 0; l < n_layers; ++l) {
        const int32_t* r = spec + l * RCN_CNN_LAYER_INTS;
        CnnLayer ly;
        ly.kind = r[0];
        ly.Hi = Hc; ly.Wi = Wc; ly.Ci = Cc;
        if (r[0] == RCN_CNN_CONV) {
            if (r[1] < 0 || r[2] < 0 || r[3] < 0) return fail(RCN_ERR_INVALID, "layer %zu: negative size", l);
            ly.Co = (size_t)r[1]; ly.kh = (size_t)r[2]; ly.kw = (size_t)r[3]; ly.padding = r[4];
            ConvShape s;
            RCN_TRY(check_conv_shape(1, Hc, Wc, Cc, ly.Co, ly.kh, ly.kw, ly.padding, &s));
            ly.Ho = s.Ho; ly.Wo = s.Wo;
            ly.w_off = off; off += ly.Co * ly.kh * ly.kw * Cc;
            ly.b_off = off; off += ly.Co;
        } else if (r[0] == RCN_CNN_POOL) {
            ly.pooling = r[1]; ly.padding = r[2];
            RCN_TRY(pool2d_shape(Hc, Wc, ly.padding, ly.pooling, &ly.Ho, &ly.Wo));
            ly.Co = Cc;
        } else {
            return fail(RCN_ERR_INVALID, "layer %zu: unknown layer kind %d", l, r[0]);
        }
        Hc = ly.Ho; Wc = ly.Wo; Cc = ly.Co;
        h->max_len = std::max(h->max_len, ly.out_len());
        h->layers.push_back(std::move(ly));
    }
    h->L = Hc * Wc * Cc;
    h->n_conv = off;
    if (h->L == 0) return fail(RCN_ERR_INVALID, "empty feature vector");
    return RCN_OK;
}

}  // namespace

extern "C" {

int rcn_cuda_cnn_create(int device, size_t H, size_t W, size_t in_channels, const int32_t* layer_spec, size_t n_layers,
                        const size_t* feedforward, size_t n_ff, size_t classes, rcn_cuda_cnn_handle* out) {
    return rcn_cuda_cnn_create_with_head(device, H, W, in_channels, layer_spec, n_layers, feedforward, n_ff, classes,
                                         RCN_HEAD_SIGMOID_QUADRATIC, out);
}

int rcn_cuda_cnn_create_with_head(int device, size_t H, size_t W, size_t in_channels, const int32_t* layer_spec, size_t n_layers,
                                  const size_t* feedforward, size_t n_ff, size_t classes, int head, rcn_cuda_cnn_handle* out) {
    if (!out) return fail(RCN_ERR_INVALID, "null out handle");
    *out = nullptr;
    if (head != RCN_HEAD_SIGMOID_QUADRATIC && head != RCN_HEAD_SOFTMAX_XENT) return fail(RCN_ERR_INVALID, "unknown head %d", head);
    if (n_layers == 0 || !layer_spec) return fail(RCN_ERR_INVALID, "the network needs at least one conv / pool layer");
    if (n_ff && !feedforward) return fail(RCN_ERR_INVALID, "null feedforward");
    if (H == 0 || W == 0 || H > 32768 || W > 32768) return fail(RCN_ERR_INVALID, "bad image size %zu x %zu", H, W);
    if (in_channels == 0) return fail(RCN_ERR_INVALID, "zero channels");
    std::unique_ptr<rcn_cuda_cnn> h(new (std::nothrow) rcn_cuda_cnn());
    if (!h) return fail(RCN_ERR_INVALID, "out of host memory");
    h->device = device;
    h->H = H; h->W = W; h->Cin = in_channels;
    RCN_TRY(plan_layers(h.get(), layer_spec, n_layers));
    std::vector<size_t> rows, cols;
    size_t n_dense = 0;
    for (size_t i = 0; i <= n_ff; ++i) {
        rows.push_back(i < n_ff ? feedforward[i] : classes);
        cols.push_back(i == 0 ? h->L : rows[i - 1]);
        if (rows[i] == 0) return fail(RCN_ERR_INVALID, "layer %zu has zero neurons", i);
        n_dense += rows[i] * cols[i] + rows[i];
    }
    h->n_params = h->n_conv + n_dense;
    // device work from here on
    rcn_cuda_model* m = nullptr;
    RCN_TRY(rcn_cuda_create(classes, nullptr, 0, feedforward, n_ff, device, &m));
    h->dense = m;
    int rc = RCN_OK;
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        rc = fail(RCN_ERR_CUDA, "cudaStreamCreateWithFlags failed");
    h->stream = h->own_stream;
    if (rc == RCN_OK) rc = rcn_cuda_set_stream(m, h->stream);
    if (rc == RCN_OK) rc = model_set_head(m, head);   // before the shapes: they pick the dense route
    if (rc == RCN_OK) rc = rcn_cuda_init_params_shapes(m, rows.data(), cols.data(), rows.size());
    if (rc == RCN_OK) rc = h->params.reserve(h->n_conv * sizeof(double));
    if (rc == RCN_OK) rc = h->grads_own.reserve(h->n_params * sizeof(double));
    if (rc == RCN_OK) rc = h->small.reserve(64);
    if (rc == RCN_OK && h->n_conv && cudaMemsetAsync(h->params.p, 0, h->n_conv * sizeof(double), h->stream) != cudaSuccess)
        rc = fail(RCN_ERR_CUDA, "cudaMemsetAsync failed");
    if (rc == RCN_OK && cudaMemsetAsync(h->grads_own.p, 0, h->n_params * sizeof(double), h->stream) != cudaSuccess)
        rc = fail(RCN_ERR_CUDA, "cudaMemsetAsync failed");
    if (rc == RCN_OK) {
        h->grads = h->grads_own.as<double>();
        rc = rcn_cuda_bind_gradient_buffer(m, h->grads + h->n_conv, n_dense);
    }
    if (rc != RCN_OK) { rcn_cuda_cnn_destroy(h.release()); return rc; }
    *out = h.release();
    return RCN_OK;
}

int rcn_cuda_cnn_destroy(rcn_cuda_cnn_handle h) {
    if (!h) return RCN_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->dense) rcn_cuda_destroy(h->dense);
    if (h->own_stream) { cudaStreamSynchronize(h->own_stream); cudaStreamDestroy(h->own_stream); }
    for (CnnLayer& ly : h->layers) { ly.out.release(); ly.argmax.release(); }
    DevBuf* bufs[] = {&h->params, &h->grads_own, &h->in_stage, &h->lab_stage, &h->out_stage, &h->x64, &h->dx, &h->gbuf[0],
                      &h->gbuf[1], &h->flip_ws, &h->wgrad_ws, &h->small, &h->rs.buf, &h->ep_chunk, &h->ep_state, &h->opt_state};
    for (DevBuf* b : bufs) b->release();
    h->oz.release();
    delete h;
    return RCN_OK;
}

int rcn_cuda_cnn_set_stream(rcn_cuda_cnn_handle h, void* cuda_stream) {
    RCN_CNN_ENTER(h);
    h->stream = (cuda_stream == RCN_STREAM_OWN) ? h->own_stream : (cudaStream_t)cuda_stream;
    return rcn_cuda_set_stream(h->dense, h->stream);
}

int rcn_cuda_cnn_synchronize(rcn_cuda_cnn_handle h) {
    RCN_CNN_ENTER(h);
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int rcn_cuda_cnn_layer_shape(rcn_cuda_cnn_handle h, size_t layer, size_t* H, size_t* W, size_t* C) {
    if (!h) return fail(RCN_ERR_INVALID, "null network handle");
    if (layer >= h->layers.size()) return fail(RCN_ERR_INVALID, "layer %zu out of range", layer);
    if (H) *H = h->layers[layer].Ho;
    if (W) *W = h->layers[layer].Wo;
    if (C) *C = h->layers[layer].Co;
    return RCN_OK;
}

int rcn_cuda_cnn_param_count(rcn_cuda_cnn_handle h, size_t* n) {
    if (!h || !n) return fail(RCN_ERR_INVALID, "null network handle / output");
    *n = h->n_params;
    return RCN_OK;
}

int rcn_cuda_cnn_set_params(rcn_cuda_cnn_handle h, const double* flat, size_t n) {
    RCN_CNN_ENTER(h);
    if (n != h->n_params) return fail(RCN_ERR_SHAPE, "network has %zu parameters, got %zu", h->n_params, n);
    if (!flat) return fail(RCN_ERR_INVALID, "null source");
    RCN_TRY(copy_in(h, h->params.as<double>(), flat, h->n_conv));
    return rcn_cuda_set_params(h->dense, flat + h->n_conv, n - h->n_conv);
}

int rcn_cuda_cnn_get_params(rcn_cuda_cnn_handle h, double* flat, size_t n) {
    RCN_CNN_ENTER(h);
    if (n != h->n_params || !flat) return fail(RCN_ERR_SHAPE, "network has %zu parameters, got %zu", h->n_params, n);
    RCN_TRY(deliver(h, flat, h->params.p, h->n_conv * sizeof(double)));
    return rcn_cuda_get_params(h->dense, flat + h->n_conv, n - h->n_conv);
}

int rcn_cuda_cnn_accumulate(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                            size_t H, size_t W) {
    RCN_CNN_ENTER(h);
    return accumulate(h, images, pixel_format, labels, B, H, W);
}

int rcn_cuda_cnn_apply(rcn_cuda_cnn_handle h, double eta, size_t global_batch) {
    RCN_CNN_ENTER(h);
    return apply(h, eta, global_batch);
}

int rcn_cuda_cnn_train_batch(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                             size_t H, size_t W, double eta) {
    RCN_CNN_ENTER(h);
    RCN_TRY(accumulate(h, images, pixel_format, labels, B, H, W));
    return apply(h, eta, B);
}

int rcn_cuda_cnn_epoch_bind(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels,
                            const int64_t* perm, size_t n_samples, size_t H, size_t W, size_t B) {
    RCN_CNN_ENTER(h);
    if (!images || !labels || B == 0 || n_samples < B)
        return fail(RCN_ERR_INVALID, "epoch_bind needs images, labels and n_samples >= B > 0");
    if (!is_device_ptr(images) || !is_device_ptr(labels) || (perm && !is_device_ptr(perm)))
        return fail(RCN_ERR_INVALID, "epoch mode needs a dataset resident in device memory");
    RCN_TRY(check_images(h, pixel_format, H, W));
    const size_t img_bytes = image_bytes(h, pixel_format);
    RCN_TRY(h->ep_chunk.reserve(B * img_bytes));
    if (pixel_format == RCN_PIXELS_U8_ROWMAJOR) RCN_TRY(h->x64.reserve(B * img_bytes * sizeof(double)));
    RCN_TRY(h->ep_state.reserve((kCnnEpSlots + B) * sizeof(int64_t)));
    RCN_CUDA_TRY(cudaMemsetAsync(h->ep_state.p, 0, (kCnnEpSlots + B) * sizeof(int64_t), h->stream));
    h->ep_images = images; h->ep_labels = labels; h->ep_perm = perm; h->ep_fmt = pixel_format;
    h->ep_n = n_samples; h->ep_B = B;
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));   // the cursor is zero before any step kernel can look at it
    return RCN_OK;
}

int rcn_cuda_cnn_epoch_seek(rcn_cuda_cnn_handle h, size_t position) {
    RCN_CNN_ENTER(h);
    RCN_TRY(require_epoch(h));
    if (position + h->ep_B > h->ep_n) return fail(RCN_ERR_INVALID, "position %zu leaves fewer than B samples", position);
    const long long pos = (long long)position;
    RCN_CUDA_TRY(cudaMemcpyAsync(h->ep_state.p, &pos, sizeof(pos), cudaMemcpyHostToDevice, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int rcn_cuda_cnn_epoch_position(rcn_cuda_cnn_handle h, size_t* position) {
    RCN_CNN_ENTER(h);
    RCN_TRY(require_epoch(h));
    if (!position) return fail(RCN_ERR_INVALID, "null output");
    long long pos = 0;
    RCN_CUDA_TRY(cudaMemcpyAsync(&pos, h->ep_state.p, sizeof(pos), cudaMemcpyDeviceToHost, h->stream));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    *position = (size_t)pos;
    return RCN_OK;
}

int rcn_cuda_cnn_epoch_accumulate(rcn_cuda_cnn_handle h) {
    RCN_CNN_ENTER(h);
    return epoch_accumulate(h);
}

int rcn_cuda_cnn_epoch_apply(rcn_cuda_cnn_handle h, double eta, size_t global_batch) {
    RCN_CNN_ENTER(h);
    return epoch_apply(h, eta, global_batch);
}

int rcn_cuda_cnn_epoch_step(rcn_cuda_cnn_handle h, double eta) {
    RCN_CNN_ENTER(h);
    RCN_TRY(epoch_accumulate(h));
    return epoch_apply(h, eta, h->ep_B);
}

int rcn_cuda_cnn_epoch_run(rcn_cuda_cnn_handle h, double eta, size_t n_steps) {
    RCN_CNN_ENTER(h);
    RCN_TRY(require_epoch(h));
    if (n_steps > (size_t)1 << 30) return fail(RCN_ERR_INVALID, "too many steps in one call");
    for (size_t k = 0; k < n_steps; ++k) {
        RCN_TRY(epoch_accumulate(h));
        RCN_TRY(epoch_apply(h, eta, h->ep_B));
    }
    return RCN_OK;
}

int rcn_cuda_cnn_last_batch_stats(rcn_cuda_cnn_handle h, double* cost, uint64_t* hits) {
    RCN_CNN_ENTER(h);
    return rcn_cuda_last_batch_stats(h->dense, cost, hits);
}

int rcn_cuda_cnn_evaluate_images(rcn_cuda_cnn_handle h, const void* images, int pixel_format, const int64_t* labels, size_t B,
                                 size_t H, size_t W, double* cost_out, uint64_t* accept_out, int64_t* labels_out) {
    RCN_CNN_ENTER(h);
    if (!cost_out || !accept_out) return fail(RCN_ERR_INVALID, "null cost / accept");
    double* st = h->small.as<double>();   // {cost, hits}
    if (B == 0) {
        RCN_CUDA_TRY(cudaMemsetAsync(st, 0, 2 * sizeof(double), h->stream));
    } else {
        const void* img = nullptr;
        const int64_t* lab = nullptr;
        bool host_in = false;
        RCN_TRY(stage_inputs(h, images, pixel_format, labels, B, H, W, &img, &lab, &host_in));
        int64_t* lab_dev = labels_out;
        const bool lab_host = labels_out && !is_device_ptr(labels_out);
        if (lab_host) { RCN_TRY(h->out_stage.reserve(B * sizeof(int64_t))); lab_dev = h->out_stage.as<int64_t>(); }
        const double* x0 = nullptr;
        RCN_TRY(forward_stack(h, img, pixel_format, B, false, false, &x0));
        RCN_TRY(model_evaluate_features(h->dense, h->layers.back().out.as<double>(), lab, B, st, lab_dev));
        if (lab_host) RCN_TRY(deliver(h, labels_out, lab_dev, B * sizeof(int64_t)));
        if (host_in) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    RCN_TRY(deliver(h, cost_out, st, sizeof(double)));
    return deliver(h, accept_out, st + 1, sizeof(uint64_t));
}

int rcn_cuda_cnn_classify_images(rcn_cuda_cnn_handle h, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                                 int64_t* labels_out) {
    RCN_CNN_ENTER(h);
    if (B == 0) return RCN_OK;
    if (!labels_out) return fail(RCN_ERR_INVALID, "null output");
    const void* img = nullptr;
    bool host_in = false;
    RCN_TRY(stage_inputs(h, images, pixel_format, nullptr, B, H, W, &img, nullptr, &host_in));
    int64_t* lab_dev = labels_out;
    const bool lab_host = !is_device_ptr(labels_out);
    if (lab_host) { RCN_TRY(h->out_stage.reserve(B * sizeof(int64_t))); lab_dev = h->out_stage.as<int64_t>(); }
    const double* x0 = nullptr;
    RCN_TRY(forward_stack(h, img, pixel_format, B, false, false, &x0));
    RCN_TRY(model_evaluate_features(h->dense, h->layers.back().out.as<double>(), nullptr, B, nullptr, lab_dev));
    if (lab_host) RCN_TRY(deliver(h, labels_out, lab_dev, B * sizeof(int64_t)));
    if (host_in) RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    return RCN_OK;
}

int rcn_cuda_cnn_bind_gradient_buffer(rcn_cuda_cnn_handle h, double* device_ptr, size_t n) {
    RCN_CNN_ENTER(h);
    if (device_ptr) {
        if (n != h->n_params) return fail(RCN_ERR_SHAPE, "gradient buffer must hold %zu doubles, got %zu", h->n_params, n);
        if (!is_device_ptr(device_ptr)) return fail(RCN_ERR_INVALID, "gradient buffer must be device memory");
    }
    double* g = device_ptr ? device_ptr : h->grads_own.as<double>();
    RCN_TRY(rcn_cuda_bind_gradient_buffer(h->dense, g + h->n_conv, h->n_params - h->n_conv));
    h->grads = g;
    return RCN_OK;
}

int rcn_cuda_cnn_gradient_buffer(rcn_cuda_cnn_handle h, double** device_ptr, size_t* n) {
    if (!h) return fail(RCN_ERR_INVALID, "null network handle");
    if (device_ptr) *device_ptr = h->grads;
    if (n) *n = h->n_params;
    return RCN_OK;
}

int rcn_cuda_cnn_get_gradients(rcn_cuda_cnn_handle h, double* flat, size_t n) {
    RCN_CNN_ENTER(h);
    if (n != h->n_params || !flat) return fail(RCN_ERR_SHAPE, "network has %zu parameters, got %zu", h->n_params, n);
    return deliver(h, flat, h->grads, n * sizeof(double));
}

int rcn_cuda_cnn_get_layer_output(rcn_cuda_cnn_handle h, size_t layer, double* out) {
    RCN_CNN_ENTER(h);
    if (layer >= h->layers.size() || !out) return fail(RCN_ERR_INVALID, "bad layer / null destination");
    if (!h->out_B) return fail(RCN_ERR_STATE, "no batch has run through the network yet");
    return deliver(h, out, h->layers[layer].out.p, h->out_B * h->layers[layer].out_len() * sizeof(double));
}

int rcn_cuda_cnn_get_input_gradient(rcn_cuda_cnn_handle h, double* out) {
    RCN_CNN_ENTER(h);
    if (!out) return fail(RCN_ERR_INVALID, "null destination");
    if (!h->grad_B) return fail(RCN_ERR_STATE, "no batch has been accumulated yet");
    return deliver(h, out, h->dx.p, h->L * h->grad_B * sizeof(double));
}

int rcn_cuda_cnn_set_optimizer(rcn_cuda_cnn_handle h, int kind, double momentum, int nesterov, double weight_decay, double beta1,
                               double beta2, double eps) {
    if (!h) return fail(RCN_ERR_INVALID, "null network handle");
    OptimConfig c;
    c.kind = kind; c.momentum = momentum; c.nesterov = nesterov; c.weight_decay = weight_decay;
    c.beta1 = beta1; c.beta2 = beta2; c.eps = eps;
    RCN_TRY(optim_validate(c));
    RCN_CUDA_TRY(cudaSetDevice(h->device));
    RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));   // no queued step still reads the old state
    h->opt_state.release();
    h->opt = OptimConfig{};
    const size_t len = optim_state_len(c, h->n_params);
    if (len) {
        RCN_TRY(h->opt_state.reserve(len * sizeof(double) + 16));
        RCN_CUDA_TRY(cudaMemsetAsync(h->opt_state.p, 0, len * sizeof(double) + 16, h->stream));
        RCN_TRY(optim_reset_state(c, h->opt_state.as<double>(), h->n_params, h->stream));
        RCN_CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->opt = c;
    alloc_generation().fetch_add(1, std::memory_order_relaxed);   // a captured step holds the old update and its arguments
    return RCN_OK;
}

int rcn_cuda_cnn_optimizer_state_size(rcn_cuda_cnn_handle h, size_t* n) {
    if (!h || !n) return fail(RCN_ERR_INVALID, "null network handle / output");
    *n = optim_state_len(h->opt, h->n_params);
    return RCN_OK;
}

int rcn_cuda_cnn_get_optimizer_state(rcn_cuda_cnn_handle h, double* state, size_t n) {
    RCN_CNN_ENTER(h);
    const size_t len = optim_state_len(h->opt, h->n_params);
    if (n != len) return fail(RCN_ERR_INVALID, "the optimizer state holds %zu doubles, got %zu", len, n);
    if (len && !state) return fail(RCN_ERR_INVALID, "null destination");
    return deliver(h, state, h->opt_state.p, len * sizeof(double));
}

int rcn_cuda_cnn_set_optimizer_state(rcn_cuda_cnn_handle h, const double* state, size_t n) {
    RCN_CNN_ENTER(h);
    const size_t len = optim_state_len(h->opt, h->n_params);
    if (n != len) return fail(RCN_ERR_INVALID, "the optimizer state holds %zu doubles, got %zu", len, n);
    if (len && !state) return fail(RCN_ERR_INVALID, "null source");
    return copy_in(h, h->opt_state.as<double>(), state, len);
}

}  // extern "C"
