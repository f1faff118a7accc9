// rcn.hpp -- C++ host side above the C ABI (include/rcn_cuda.h), mirroring the public API of the reference crate
// `rcn` (jtstrader/mercer-research): same names, argument meaning and error behaviour, so that host code and tests read
// like the reference's own.  Header-only, C++17, depends on nothing but the C header; link with -lrcn_cuda.
//
//   reference (rcn/src/...)                                    here
//   utils/kernel.rs:16-35   SeparableOperator, Padding, Pooling    rcn::SeparableOperator, rcn::Padding, rcn::Pooling
//   utils/kernel.rs:38-53   sobel_separated                        rcn::sobel_separated
//   utils/kernel.rs:61-100  trait Convolve2D on a matrix           DMatrix::convolve_2d / convolve_2d_separated / relu
//   utils/kernel.rs:219-236 trait Pool2D                           DMatrix::pool_2d
//   rcn.rs:28-31            Weights, Bias                          rcn::Weights, rcn::Bias
//   rcn.rs:35-38            RCNLayer                               rcn::RCNLayer
//   rcn.rs:58-64,82,126-133 RCN::new / classify / train            rcn::RCN (train / classify take decoded pixels)
//
// Where the reference panics on a contract violation (kernel.rs:127,133,156,200,247,280,284; nalgebra dimension
// mismatch) this layer throws rcn::Error carrying the library's status code and the reference's message.  There is no
// CPU fallback: without a CUDA device every compute call throws with status RCN_ERR_CUDA.
//
// PNG decoding is the `image` crate's job in the reference (rcn.rs:83,394-398) and stays outside the accelerated path:
// the caller hands decoded grayscale pixels (GraySet), or binary PGM files to classify_pgm().
#pragma once

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <numeric>
#include <ostream>
#include <random>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "rcn_cuda.h"

namespace rcn {

/// A reference `panic!` (or a CUDA failure) surfaced by the C ABI.
struct Error : std::runtime_error {
    int status;
    Error(int status_, const std::string& msg) : std::runtime_error(msg), status(status_) {}
};

inline void check(int rc) {
    if (rc != RCN_OK) {
        const char* msg = rcn_cuda_last_error();
        throw Error(rc, msg ? msg : "rcn_cuda call failed");
    }
}

enum class SeparableOperator { Top = RCN_OP_TOP, Bottom = RCN_OP_BOTTOM, Left = RCN_OP_LEFT, Right = RCN_OP_RIGHT };  // kernel.rs:16-21
enum class Padding { None = RCN_PADDING_NONE, Same = RCN_PADDING_SAME };                                                // kernel.rs:25-28
enum class Pooling { Average = RCN_POOLING_AVERAGE, Max = RCN_POOLING_MAX };                                            // kernel.rs:32-35

/// nalgebra's DMatrix<f64>: column-major storage (element (r, c) at data[c * nrows + r]), owned.
class DMatrix {
  public:
    DMatrix() = default;
    DMatrix(size_t nrows, size_t ncols) : nrows_(nrows), ncols_(ncols), data_(nrows * ncols, 0.0) {}
    static DMatrix zeros(size_t nrows, size_t ncols) { return DMatrix(nrows, ncols); }
    /// DMatrix::from_row_iterator / from_row_slice: values given row by row.
    template <typename It>
    static DMatrix from_row_iterator(size_t nrows, size_t ncols, It it) {
        DMatrix m(nrows, ncols);
        for (size_t r = 0; r < nrows; ++r)
            for (size_t c = 0; c < ncols; ++c, ++it) m(r, c) = static_cast<double>(*it);
        return m;
    }
    static DMatrix from_row_slice(size_t nrows, size_t ncols, std::initializer_list<double> v) {
        if (v.size() != nrows * ncols) throw std::invalid_argument("from_row_slice: wrong number of elements");
        return from_row_iterator(nrows, ncols, v.begin());
    }
    /// DMatrix::from_vec: column-major values taken as they are.
    static DMatrix from_vec(size_t nrows, size_t ncols, std::vector<double> v) {
        if (v.size() != nrows * ncols) throw std::invalid_argument("from_vec: wrong number of elements");
        DMatrix m;
        m.nrows_ = nrows; m.ncols_ = ncols; m.data_ = std::move(v);
        return m;
    }
    size_t nrows() const { return nrows_; }
    size_t ncols() const { return ncols_; }
    std::pair<size_t, size_t> shape() const { return {nrows_, ncols_}; }
    size_t len() const { return data_.size(); }
    double& operator()(size_t r, size_t c) { return data_[c * nrows_ + r]; }
    double operator()(size_t r, size_t c) const { return data_[c * nrows_ + r]; }
    const double* as_ptr() const { return data_.data(); }
    double* as_mut_ptr() { return data_.data(); }
    const std::vector<double>& as_slice() const { return data_; }
    bool operator==(const DMatrix& o) const { return nrows_ == o.nrows_ && ncols_ == o.ncols_ && data_ == o.data_; }
    bool operator!=(const DMatrix& o) const { return !(*this == o); }
    /// Matrix product (only what the reference's own tests need: the 3x1 * 1x3 Sobel factors, kernel.rs:400-417).
    DMatrix operator*(const DMatrix& o) const {
        if (ncols_ != o.nrows_) throw std::invalid_argument("matrix product: dimension mismatch");
        DMatrix out(nrows_, o.ncols_);
        for (size_t c = 0; c < o.ncols_; ++c)
            for (size_t k = 0; k < ncols_; ++k)
                for (size_t r = 0; r < nrows_; ++r) out(r, c) += (*this)(r, k) * o(k, c);
        return out;
    }

    // ---- trait Convolve2D (kernel.rs:61-100): computed on the GPU `device` --------------------------------------------
    /// 2-D cross-correlation with an arbitrary kernel (kernel.rs:110-194), including the reference's SAME-padding copy.
    DMatrix convolve_2d(const DMatrix& kernel, Padding padding, int device = 0) const {
        size_t oh = nrows_, ow = ncols_;
        if (padding == Padding::None) {   // (H - kh + 1) x (W - kw + 1); an oversized kernel is reported by the library
            oh = nrows_ + 1 > kernel.nrows_ ? nrows_ + 1 - kernel.nrows_ : 0;
            ow = ncols_ + 1 > kernel.ncols_ ? ncols_ + 1 - kernel.ncols_ : 0;
        }
        DMatrix out(oh, ow);
        double none = 0.0;   // an oversized kernel leaves nothing to write: the library must still see a non-null output
        check(rcn_cuda_convolve_2d(device, nullptr, as_ptr(), nrows_, ncols_, kernel.as_ptr(), kernel.nrows_, kernel.ncols_,
                                   static_cast<int>(padding), out.len() ? out.as_mut_ptr() : &none));
        return out;
    }
    /// relu(conv(conv(X, v), h)) with the separated Sobel factors of `op` (kernel.rs:196-207).
    DMatrix convolve_2d_separated(SeparableOperator op, Padding padding, int device = 0) const {
        const bool same = padding == Padding::Same;
        DMatrix out(same ? nrows_ : (nrows_ > 2 ? nrows_ - 2 : 0), same ? ncols_ : (ncols_ > 2 ? ncols_ - 2 : 0));
        double none = 0.0;
        check(rcn_cuda_convolve_2d_separated(device, nullptr, as_ptr(), nrows_, ncols_, static_cast<int>(op),
                                             static_cast<int>(padding), out.len() ? out.as_mut_ptr() : &none));
        return out;
    }
    /// kernel.rs:209-216
    DMatrix relu(int device = 0) const {
        DMatrix out(nrows_, ncols_);
        check(rcn_cuda_relu(device, nullptr, as_ptr(), len(), out.as_mut_ptr()));
        return out;
    }
    // ---- trait Pool2D (kernel.rs:219-236) -----------------------------------------------------------------------------
    /// 2x2 window, stride 2 (kernel.rs:245-349); `argmax` (optional) receives 2*dy+dx of the winning element, last maximal
    /// element wins -- an extension, the reference returns values only.
    DMatrix pool_2d(Padding padding, Pooling pooling, std::vector<uint8_t>* argmax = nullptr, int device = 0) const {
        const bool same = padding == Padding::Same;
        DMatrix out(same ? (nrows_ + 1) / 2 : nrows_ / 2, same ? (ncols_ + 1) / 2 : ncols_ / 2);
        if (argmax) argmax->assign(out.len(), 0);
        double none = 0.0;
        check(rcn_cuda_pool_2d(device, nullptr, as_ptr(), nrows_, ncols_, static_cast<int>(padding), static_cast<int>(pooling),
                               out.len() ? out.as_mut_ptr() : &none, argmax && out.len() ? argmax->data() : nullptr));
        return out;
    }

  private:
    size_t nrows_ = 0, ncols_ = 0;
    std::vector<double> data_;
};

/// kernel.rs:38-53: (3x1 vertical factor, 1x3 horizontal factor) of a Sobel operator.
inline std::pair<DMatrix, DMatrix> sobel_separated(SeparableOperator op) {
    switch (op) {
        case SeparableOperator::Top: return {DMatrix::from_row_slice(3, 1, {1, 0, -1}), DMatrix::from_row_slice(1, 3, {1, 2, 1})};
        case SeparableOperator::Bottom: return {DMatrix::from_row_slice(3, 1, {-1, 0, 1}), DMatrix::from_row_slice(1, 3, {1, 2, 1})};
        case SeparableOperator::Left: return {DMatrix::from_row_slice(3, 1, {1, 2, 1}), DMatrix::from_row_slice(1, 3, {1, 0, -1})};
        default: return {DMatrix::from_row_slice(3, 1, {1, 2, 1}), DMatrix::from_row_slice(1, 3, {-1, 0, 1})};
    }
}

/// rcn.rs:35-38
struct RCNLayer {
    int code;   // RCN_LAYER_{CONV_NONE, CONV_SAME, POOL_AVERAGE, POOL_MAX}
    static RCNLayer Convolve2D(Padding p) { return {static_cast<int>(p)}; }
    static RCNLayer Pool2D(Pooling p) { return {2 + static_cast<int>(p)}; }
};

/// rcn.rs:28-31
struct Weights { DMatrix m; };
struct Bias { std::vector<double> v; };

/// N decoded grayscale images of h x w bytes, row-major (the `image` crate's Luma8 buffer), with their class indices.
struct GraySet {
    std::vector<uint8_t> pixels;
    std::vector<int64_t> labels;
    size_t n = 0, h = 0, w = 0;
};

/// Reads a binary PGM (P5, maxval <= 255): the one image format this header decodes itself.
inline bool read_pgm(const std::string& path, std::vector<uint8_t>* pixels, size_t* h, size_t* w) {
    std::ifstream f(path, std::ios::binary);
    std::string magic;
    size_t ww = 0, hh = 0, maxval = 0;
    auto token = [&](std::string* out) {
        out->clear();
        int c;
        while ((c = f.get()) != EOF) {
            if (c == '#') { while ((c = f.get()) != EOF && c != '\n') {} continue; }
            if (c == ' ' || c == '\t' || c == '\r' || c == '\n') { if (!out->empty()) return; continue; }
            out->push_back(static_cast<char>(c));
        }
    };
    std::string t;
    token(&magic);
    if (magic != "P5") return false;
    try {
        token(&t); ww = std::stoul(t);
        token(&t); hh = std::stoul(t);
        token(&t); maxval = std::stoul(t);
    } catch (const std::exception&) { return false; }
    if (!ww || !hh || maxval > 255) return false;
    pixels->resize(ww * hh);
    f.read(reinterpret_cast<char*>(pixels->data()), static_cast<std::streamsize>(pixels->size()));
    if (static_cast<size_t>(f.gcount()) != pixels->size()) return false;
    *h = hh; *w = ww;
    return true;
}

/// rcn.rs:13-25, 58-64: the model. Parameters live in HBM behind the handle; move-only like a Rust value.
class RCN {
  public:
    /// RCN::new (rcn.rs:58-64). The paths are kept for parity with the reference's struct (they are part of `rcn.bin`).
    RCN(size_t classes, std::vector<RCNLayer> convpool_cfg, std::vector<size_t> feedforward_cfg, std::string training_path = "",
        std::string testing_path = "", int device = 0)
        : classes_(classes), convpool_cfg_(std::move(convpool_cfg)), feedforward_cfg_(std::move(feedforward_cfg)),
          training_path_(std::move(training_path)), testing_path_(std::move(testing_path)), device_(device) {
        std::vector<int32_t> codes;
        for (const RCNLayer& l : convpool_cfg_) codes.push_back(l.code);
        check(rcn_cuda_create(classes_, codes.data(), codes.size(), feedforward_cfg_.data(), feedforward_cfg_.size(), device_, &h_));
    }
    ~RCN() { if (h_) rcn_cuda_destroy(h_); }
    RCN(const RCN&) = delete;
    RCN& operator=(const RCN&) = delete;
    RCN(RCN&& o) noexcept { *this = std::move(o); }
    RCN& operator=(RCN&& o) noexcept {
        if (this != &o) {
            if (h_) rcn_cuda_destroy(h_);
            h_ = o.h_; o.h_ = nullptr;
            classes_ = o.classes_; device_ = o.device_;
            convpool_cfg_ = std::move(o.convpool_cfg_); feedforward_cfg_ = std::move(o.feedforward_cfg_);
            training_path_ = std::move(o.training_path_); testing_path_ = std::move(o.testing_path_);
        }
        return *this;
    }

    rcn_cuda_handle handle() const { return h_; }
    size_t classes() const { return classes_; }
    const std::string& training_path() const { return training_path_; }
    const std::string& testing_path() const { return testing_path_; }

    // ---- shapes / parameters ------------------------------------------------------------------------------------------
    /// Length of flatten_feature_set's output for an h x w image (rcn.rs:317-356).
    size_t feature_len(size_t h, size_t w) const {
        size_t maps = 0, mh = 0, mw = 0;
        check(rcn_cuda_feature_shape(h_, h, w, &maps, &mh, &mw));
        return maps * mh * mw;
    }
    /// Number of dense layers; 0 while the model has no parameters yet (`layer_weights.is_empty()`, rcn.rs:139).
    size_t num_layers() const {
        size_t n = 0;
        const int rc = rcn_cuda_num_layers(h_, &n);
        if (rc == RCN_ERR_STATE) return 0;
        check(rc);
        return n;
    }
    std::pair<size_t, size_t> layer_shape(size_t layer) const {
        size_t r = 0, c = 0;
        check(rcn_cuda_layer_shape(h_, layer, &r, &c));
        return {r, c};
    }
    /// load_weights_and_bias (rcn.rs:425-457, 500-523): the reference's shapes -- including its `4^c / 2^p * l` first
    /// width -- filled with unscaled N(0, 1) draws in column-major order. The reference's generator is unseeded; here
    /// the caller owns the seed.
    void load_weights_and_bias(size_t l, uint64_t seed) {
        check(rcn_cuda_init_params(h_, l));
        std::mt19937_64 gen(seed);
        std::normal_distribution<double> n01(0.0, 1.0);
        for (size_t layer = 0; layer < num_layers(); ++layer) {
            auto [r, c] = layer_shape(layer);
            std::vector<double> w(r * c), b(r);
            for (double& x : w) x = n01(gen);
            for (double& x : b) x = n01(gen);
            check(rcn_cuda_set_weights(h_, layer, r, c, w.data()));
            check(rcn_cuda_set_bias(h_, layer, r, b.data()));
        }
    }
    /// Shapes only (zeroed parameters), for callers that inject values with set_weights / set_bias.
    void init_params(size_t l) { check(rcn_cuda_init_params(h_, l)); }
    Weights layer_weights(size_t layer) const {
        auto [r, c] = layer_shape(layer);
        Weights w{DMatrix(r, c)};
        check(rcn_cuda_get_weights(h_, layer, w.m.as_mut_ptr()));
        return w;
    }
    Bias layer_bias(size_t layer) const {
        Bias b{std::vector<double>(layer_shape(layer).first)};
        check(rcn_cuda_get_bias(h_, layer, b.v.data()));
        return b;
    }
    void set_weights(size_t layer, const DMatrix& w) { check(rcn_cuda_set_weights(h_, layer, w.nrows(), w.ncols(), w.as_ptr())); }
    void set_bias(size_t layer, const std::vector<double>& b) { check(rcn_cuda_set_bias(h_, layer, b.size(), b.data())); }
    std::pair<double, double> scale_set() const {
        double m = 0, s = 0;
        check(rcn_cuda_get_scale(h_, &m, &s));
        return {m, s};
    }
    void set_scale_set(std::pair<double, double> ms) { check(rcn_cuda_set_scale(h_, ms.first, ms.second)); }

    // ---- inference ----------------------------------------------------------------------------------------------------
    /// RCN::classify (rcn.rs:82-98) on decoded pixels: features, standardise with scale_set, forward, argmax (last max wins).
    size_t classify(const uint8_t* pixels, size_t h, size_t w) const {
        int64_t label = 0;
        check(rcn_cuda_classify(h_, pixels, RCN_PIXELS_U8_ROWMAJOR, 1, h, w, &label));
        return static_cast<size_t>(label);
    }
    std::vector<int64_t> classify(const GraySet& set) const {
        std::vector<int64_t> labels(set.n);
        if (set.n) check(rcn_cuda_classify(h_, set.pixels.data(), RCN_PIXELS_U8_ROWMAJOR, set.n, set.h, set.w, labels.data()));
        return labels;
    }
    /// Test-set evaluation (rcn.rs:152-157) of a decoded set standardised with scale_set: {accept, quadratic cost
    /// sum_b 0.5*|a - y|^2}, with the exact-one-hot hit rule of the reference's epoch loop.
    std::pair<uint64_t, double> evaluate_images(const GraySet& set) const {
        uint64_t accept = 0;
        double cost = 0.0;
        check(rcn_cuda_evaluate_images(h_, set.pixels.data(), RCN_PIXELS_U8_ROWMAJOR, set.labels.data(), set.n, set.h, set.w,
                                       &cost, &accept, nullptr));
        return {accept, cost};
    }
    /// classify(img_path) for a binary PGM; an unreadable file is an error value like the reference's `?` (rcn.rs:83).
    size_t classify_pgm(const std::string& img_path) const {
        std::vector<uint8_t> px;
        size_t h = 0, w = 0;
        if (!read_pgm(img_path, &px, &h, &w)) throw std::runtime_error("cannot decode " + img_path + " (binary PGM expected)");
        return classify(px.data(), h, w);
    }
    /// classify_test (rcn.rs:105-116) on one standardised feature vector: the activations of the last layer.
    std::vector<double> classify_test(const std::vector<double>& x) const {
        std::vector<double> out(classes_);
        check(rcn_cuda_forward(h_, x.data(), 1, out.data()));
        return out;
    }

    // ---- training -----------------------------------------------------------------------------------------------------
    /// train_batch (rcn.rs:176-223) on standardised feature vectors (B x n_in, sample-contiguous) with one-hot targets.
    void train_batch(const std::vector<double>& feats, const std::vector<double>& onehot, size_t batch, double eta) {
        check(rcn_cuda_train_batch(h_, feats.data(), onehot.data(), nullptr, batch, eta));
    }
    /// RCN::train (rcn.rs:126-167) on decoded sets: statistics of each set in turn (scale_set ends up holding the TEST
    /// set's, rcn.rs:134-137,406, and the training steps standardise with the training set's), parameters drawn if absent
    /// (rcn.rs:139-141), per epoch a shuffle (rcn.rs:146), the chunks_exact loop (rcn.rs:147-149: one call, remainder
    /// dropped), the evaluation with the exact-one-hot rule (rcn.rs:152-157) and the reference's log line (rcn.rs:158-164).
    /// Returns the per-epoch accept counts.
    std::vector<uint64_t> train(const GraySet& training, const GraySet& testing, size_t batch_size, size_t epochs, double eta,
                                uint64_t seed = 0, std::ostream* log = nullptr) {
        if (!training.n || !testing.n) throw std::invalid_argument("train: empty data set");
        const auto train_scale = gen_scales(training);
        const auto test_scale = gen_scales(testing);
        const size_t l = feature_len(training.h, training.w);
        if (num_layers() == 0) load_weights_and_bias(l, seed);
        // test features, standardised with the test statistics, computed once
        set_scale_set(test_scale);
        std::vector<double> test_feats(feature_len(testing.h, testing.w) * testing.n);
        check(rcn_cuda_features(h_, testing.pixels.data(), RCN_PIXELS_U8_ROWMAJOR, testing.n, testing.h, testing.w, 1, test_feats.data()));
        const size_t img = training.h * training.w;
        std::vector<size_t> order(training.n);
        std::iota(order.begin(), order.end(), size_t{0});
        std::vector<uint8_t> shuffled(training.n * img);
        std::vector<int64_t> shuffled_labels(training.n);
        std::mt19937_64 gen(seed ^ 0x9E3779B97F4A7C15ull);
        std::vector<uint64_t> history;
        for (size_t e = 0; e < epochs; ++e) {
            std::shuffle(order.begin(), order.end(), gen);
            for (size_t dst = 0; dst < training.n; ++dst) {
                std::copy_n(training.pixels.data() + order[dst] * img, img, shuffled.data() + dst * img);
                shuffled_labels[dst] = training.labels[order[dst]];
            }
            set_scale_set(train_scale);
            size_t steps = 0;
            check(rcn_cuda_train_epoch_host(h_, shuffled.data(), RCN_PIXELS_U8_ROWMAJOR, shuffled_labels.data(), training.n,
                                            training.h, training.w, batch_size, eta, 0, nullptr, nullptr, &steps));
            set_scale_set(test_scale);
            uint64_t accept = 0;
            check(rcn_cuda_evaluate(h_, test_feats.data(), testing.labels.data(), testing.n, &accept));
            history.push_back(accept);
            if (log) {
                char line[128];
                std::snprintf(line, sizeof(line), "Epoch %zu: %llu/%zu [%.2f%%]", e, static_cast<unsigned long long>(accept),
                              testing.n, static_cast<double>(accept) / static_cast<double>(testing.n) * 100.0);
                *log << line << "\n";
            }
        }
        return history;
    }

    /// gen_scales (rcn.rs:230-251) over the raw features of a whole set; also stored as scale_set.
    std::pair<double, double> gen_scales(const GraySet& set) {
        const size_t l = feature_len(set.h, set.w);
        std::vector<double> feats(l * set.n);
        check(rcn_cuda_features(h_, set.pixels.data(), RCN_PIXELS_U8_ROWMAJOR, set.n, set.h, set.w, 0, feats.data()));
        double mean = 0, sd = 0;
        check(rcn_cuda_gen_scales(h_, feats.data(), l, set.n, &mean, &sd));
        return {mean, sd};
    }

  private:
    rcn_cuda_handle h_ = nullptr;
    size_t classes_ = 0;
    std::vector<RCNLayer> convpool_cfg_;
    std::vector<size_t> feedforward_cfg_;
    std::string training_path_, testing_path_;
    int device_ = 0;
};

/// Output head of a ConvNet's dense stack (RCN_HEAD_* in rcn_cuda.h): the reference's sigmoid layer with quadratic cost, or an
/// affine output layer with softmax and cross-entropy.
enum class Head : int { SigmoidQuadratic = RCN_HEAD_SIGMOID_QUADRATIC, SoftmaxCrossEntropy = RCN_HEAD_SOFTMAX_XENT };

/// Optimizer of a ConvNet's update (rcn_cuda_cnn_set_optimizer in rcn_cuda.h gives the formulas); the other kind's fields are
/// ignored.  Optimizer{} is plain SGD, the default update.
struct Optimizer {
    int kind = RCN_OPTIMIZER_SGD;
    double momentum = 0.0;
    bool nesterov = false;
    double weight_decay = 0.0;
    double beta1 = 0.9, beta2 = 0.999, eps = 1e-8;

    static Optimizer sgd(double momentum = 0.0, bool nesterov = false, double weight_decay = 0.0) {
        Optimizer o;
        o.momentum = momentum;
        o.nesterov = nesterov;
        o.weight_decay = weight_decay;
        return o;
    }
    static Optimizer adamw(double beta1 = 0.9, double beta2 = 0.999, double eps = 1e-8, double weight_decay = 0.0) {
        Optimizer o;
        o.kind = RCN_OPTIMIZER_ADAMW;
        o.beta1 = beta1;
        o.beta2 = beta2;
        o.eps = eps;
        o.weight_decay = weight_decay;
        return o;
    }
};

/// Learned conv / pool layers in front of the reference's dense stack (rcn_cuda_cnn_* in rcn_cuda.h): a thin owner of the
/// handle.  Images are u8 (B, H, W) row-major or f64 (B, H, W, C) NHWC, host or device memory.
class ConvNet {
  public:
    struct Layer {
        static Layer conv(size_t co, size_t kh, size_t kw, Padding p) {
            return Layer{{RCN_CNN_CONV, (int32_t)co, (int32_t)kh, (int32_t)kw, (int32_t)p}};
        }
        static Layer pool(Pooling pooling, Padding p) { return Layer{{RCN_CNN_POOL, (int32_t)pooling, (int32_t)p, 0, 0}}; }
        int32_t spec[RCN_CNN_LAYER_INTS];
    };

    ConvNet(size_t H, size_t W, size_t in_channels, const std::vector<Layer>& layers, const std::vector<size_t>& feedforward,
            size_t classes, int device = 0, Head head = Head::SigmoidQuadratic) {
        std::vector<int32_t> spec;
        for (const Layer& l : layers) spec.insert(spec.end(), l.spec, l.spec + RCN_CNN_LAYER_INTS);
        check(rcn_cuda_cnn_create_with_head(device, H, W, in_channels, spec.data(), layers.size(), feedforward.data(),
                                            feedforward.size(), classes, (int)head, &h_));
    }
    ~ConvNet() { rcn_cuda_cnn_destroy(h_); }
    ConvNet(const ConvNet&) = delete;
    ConvNet& operator=(const ConvNet&) = delete;

    size_t n_params() const {
        size_t n = 0;
        check(rcn_cuda_cnn_param_count(h_, &n));
        return n;
    }
    void set_params(const std::vector<double>& flat) { check(rcn_cuda_cnn_set_params(h_, flat.data(), flat.size())); }
    std::vector<double> get_params() const {
        std::vector<double> p(n_params());
        check(rcn_cuda_cnn_get_params(h_, p.data(), p.size()));
        return p;
    }
    std::vector<double> get_gradients() const {
        std::vector<double> g(n_params());
        check(rcn_cuda_cnn_get_gradients(h_, g.data(), g.size()));
        return g;
    }
    void train_batch(const void* images, int pixel_format, const int64_t* labels, size_t B, size_t H, size_t W, double eta) {
        check(rcn_cuda_cnn_train_batch(h_, images, pixel_format, labels, B, H, W, eta));
    }
    void accumulate(const void* images, int pixel_format, const int64_t* labels, size_t B, size_t H, size_t W) {
        check(rcn_cuda_cnn_accumulate(h_, images, pixel_format, labels, B, H, W));
    }
    void apply(double eta, size_t global_batch) { check(rcn_cuda_cnn_apply(h_, eta, global_batch)); }
    /// (quadratic cost, hit count) of the last accumulated batch under the pre-update parameters.
    std::pair<double, uint64_t> last_batch_stats() const {
        double c = 0.0;
        uint64_t hits = 0;
        check(rcn_cuda_cnn_last_batch_stats(h_, &c, &hits));
        return {c, hits};
    }
    /// (accept, cost) of a labelled batch (rcn.rs:152-157 rule); labels_out (optional) receives the predictions.
    std::pair<uint64_t, double> evaluate(const void* images, int pixel_format, const int64_t* labels, size_t B, size_t H, size_t W,
                                         int64_t* labels_out = nullptr) {
        double c = 0.0;
        uint64_t acc = 0;
        check(rcn_cuda_cnn_evaluate_images(h_, images, pixel_format, labels, B, H, W, &c, &acc, labels_out));
        return {acc, c};
    }
    std::vector<int64_t> classify(const void* images, int pixel_format, size_t B, size_t H, size_t W) {
        std::vector<int64_t> out(B);
        check(rcn_cuda_cnn_classify_images(h_, images, pixel_format, B, H, W, out.data()));
        return out;
    }
    /// Epoch mode over a dataset in DEVICE memory (rcn_cuda_cnn_epoch_* in rcn_cuda.h); perm may be null (identity).
    void epoch_bind(const void* images, int pixel_format, const int64_t* labels, const int64_t* perm, size_t n_samples,
                    size_t H, size_t W, size_t B) {
        check(rcn_cuda_cnn_epoch_bind(h_, images, pixel_format, labels, perm, n_samples, H, W, B));
    }
    void epoch_seek(size_t position) { check(rcn_cuda_cnn_epoch_seek(h_, position)); }
    size_t epoch_position() const {
        size_t p = 0;
        check(rcn_cuda_cnn_epoch_position(h_, &p));
        return p;
    }
    void epoch_accumulate() { check(rcn_cuda_cnn_epoch_accumulate(h_)); }
    void epoch_apply(double eta, size_t global_batch) { check(rcn_cuda_cnn_epoch_apply(h_, eta, global_batch)); }
    void epoch_step(double eta) { check(rcn_cuda_cnn_epoch_step(h_, eta)); }
    void epoch_run(double eta, size_t n_steps) { check(rcn_cuda_cnn_epoch_run(h_, eta, n_steps)); }
    /// Selects the update of apply / epoch_apply and resets its state (captured steps must be re-captured).
    void set_optimizer(const Optimizer& o) {
        check(rcn_cuda_cnn_set_optimizer(h_, o.kind, o.momentum, o.nesterov ? 1 : 0, o.weight_decay, o.beta1, o.beta2, o.eps));
    }
    /// The optimizer's state as a flat vector (empty for plain SGD), to resume training in another network.
    std::vector<double> optimizer_state() const {
        size_t n = 0;
        check(rcn_cuda_cnn_optimizer_state_size(h_, &n));
        std::vector<double> s(n);
        check(rcn_cuda_cnn_get_optimizer_state(h_, s.data(), n));
        return s;
    }
    void set_optimizer_state(const std::vector<double>& s) { check(rcn_cuda_cnn_set_optimizer_state(h_, s.data(), s.size())); }
    rcn_cuda_cnn_handle handle() const { return h_; }

  private:
    rcn_cuda_cnn_handle h_ = nullptr;
};

}  // namespace rcn
