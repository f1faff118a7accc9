// C++ host tests above the C ABI (include/rcn.hpp): the reference crate's own unit tests (rcn/src/utils/kernel.rs:352-441,
// rcn/src/rcn.rs:525-538) restated against the C++ mirror of its API, plus the derived known-answer vectors of SURVEY.md
// Appendix B.  `host_test cpu [dir]` needs no GPU (host-side checks, contract violations, the no-fallback rule) and writes
// its scratch files under `dir` (default /tmp); `host_test gpu` runs the compute cases on cuda:0.  Exit code 0 and a final
// "... ok" line on success.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>

#include "rcn.hpp"

using rcn::DMatrix;
using rcn::Padding;
using rcn::Pooling;
using rcn::SeparableOperator;

static int g_failed = 0;
#define EXPECT(cond)                                                                      \
    do {                                                                                  \
        if (!(cond)) { std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); ++g_failed; } \
    } while (0)

template <typename F>
static int status_of(F&& f) {
    try { f(); } catch (const rcn::Error& e) { return e.status; }
    return RCN_OK;
}

static bool close(double got, double want, double rtol = 1e-12) { return std::fabs(got - want) <= rtol * std::max(1.0, std::fabs(want)); }

// kernel.rs:400-417
static void verify_separated_sobels() {
    const DMatrix top = DMatrix::from_row_slice(3, 3, {1, 2, 1, 0, 0, 0, -1, -2, -1});
    const DMatrix bottom = DMatrix::from_row_slice(3, 3, {-1, -2, -1, 0, 0, 0, 1, 2, 1});
    const DMatrix left = DMatrix::from_row_slice(3, 3, {1, 0, -1, 2, 0, -2, 1, 0, -1});
    const DMatrix right = DMatrix::from_row_slice(3, 3, {-1, 0, 1, -2, 0, 2, -1, 0, 1});
    auto product = [](SeparableOperator op) { auto vh = rcn::sobel_separated(op); return vh.first * vh.second; };
    EXPECT(top == product(SeparableOperator::Top));
    EXPECT(left == product(SeparableOperator::Left));
    EXPECT(right == product(SeparableOperator::Right));
    EXPECT(bottom == product(SeparableOperator::Bottom));
}

// kernel.rs:419-432
static void validate_padding_calc() {
    const size_t m0 = 28, m1 = 28, k0 = 3, k1 = 3;
    const size_t r0 = m0 - k0 + 1, r1 = m1 - k1 + 1;
    EXPECT(m0 - r0 < k0);
    EXPECT(m1 - r1 < k1);
}

static int run_cpu(const std::string& dir) {
    verify_separated_sobels();
    validate_padding_calc();
    // no CPU fallback: without a device the model cannot even be created
    try {
        rcn::RCN model(10, {rcn::RCNLayer::Convolve2D(Padding::Same), rcn::RCNLayer::Pool2D(Pooling::Max)}, {30});
        std::printf("note: a CUDA device is present, skipping the no-device check\n");
    } catch (const rcn::Error& e) {
        EXPECT(e.status == RCN_ERR_CUDA);
        EXPECT(std::strstr(e.what(), "no CPU fallback") != nullptr);
    }
    // contract violations are reported before any device work, with the reference's panic classes
    EXPECT(status_of([] { DMatrix(2, 5).convolve_2d_separated(SeparableOperator::Top, Padding::Same); }) == RCN_ERR_SHAPE);     // kernel.rs:199-201
    EXPECT(status_of([] { DMatrix(1, 5).pool_2d(Padding::Same, Pooling::Max); }) == RCN_ERR_SHAPE);                            // kernel.rs:246-251
    EXPECT(status_of([] { DMatrix(4, 4).pool_2d(Padding::Same, Pooling::Average); }) == RCN_ERR_NOT_IMPLEMENTED);              // kernel.rs:283-285
    EXPECT(status_of([] { DMatrix(4, 4).convolve_2d(DMatrix(2, 2), Padding::Same); }) == RCN_ERR_SHAPE);                       // kernel.rs:131-135
    EXPECT(status_of([] { DMatrix(2, 2).convolve_2d(DMatrix(3, 3), Padding::None); }) == RCN_ERR_SHAPE);                       // kernel.rs:123-128
    EXPECT(status_of([] { DMatrix(8, 8).convolve_2d(DMatrix(5, 5), Padding::Same); }) == RCN_ERR_OUT_OF_BOUNDS);               // kernel.rs:156
    EXPECT(rcn::RCNLayer::Convolve2D(Padding::Same).code == RCN_LAYER_CONV_SAME && rcn::RCNLayer::Pool2D(Pooling::Max).code == RCN_LAYER_POOL_MAX);
    // column-major storage and the row-iterator constructor (lib.rs:29-33 builds the pixel matrix the same way)
    {
        const DMatrix m = DMatrix::from_row_slice(2, 3, {1, 2, 3, 4, 5, 6});
        EXPECT(m(0, 2) == 3 && m(1, 0) == 4 && m.as_slice() == std::vector<double>({1, 4, 2, 5, 3, 6}));
        EXPECT(DMatrix::from_vec(2, 3, {1, 4, 2, 5, 3, 6}) == m && m.shape() == std::make_pair(size_t{2}, size_t{3}));
    }
    // the one image format the header decodes itself: binary PGM, comments allowed, 16-bit and truncated files rejected
    {
        const std::string path = dir + "/rcn_host_test.pgm";
        { std::ofstream f(path, std::ios::binary); f << "P5\n# a comment\n3 2\n255\n"; f.write("\x00\x01\x02\xfd\xfe\xff", 6); }
        std::vector<uint8_t> px;
        size_t h = 0, w = 0;
        EXPECT(rcn::read_pgm(path, &px, &h, &w) && h == 2 && w == 3 && px == std::vector<uint8_t>({0, 1, 2, 253, 254, 255}));
        { std::ofstream f(path, std::ios::binary); f << "P5\n3 2\n65535\n"; f.write("\0\0\0\0\0\0\0\0\0\0\0\0", 12); }
        EXPECT(!rcn::read_pgm(path, &px, &h, &w));
        { std::ofstream f(path, std::ios::binary); f << "P5\n3 2\n255\n"; f.write("\x00\x01", 2); }
        EXPECT(!rcn::read_pgm(path, &px, &h, &w));
        { std::ofstream f(path, std::ios::binary); f << "P2\n3 2\n255\n1 2 3 4 5 6\n"; }
        EXPECT(!rcn::read_pgm(path, &px, &h, &w));
        EXPECT(!rcn::read_pgm(dir + "/rcn_host_test_missing.pgm", &px, &h, &w));
        std::remove(path.c_str());
    }
    if (!g_failed) std::printf("cpu ok\n");
    return g_failed ? 1 : 0;
}

// SURVEY.md Appendix B
static const double X65[30] = {8, 6, 5, 2, 3, 0, 0, 0, 1, 8, 6, 9, 5, 6, 9, 7, 6, 5, 5, 9, 2, 8, 6, 0, 3, 8, 5, 0, 7, 7};
struct Kat { SeparableOperator op; double conv[30]; double pool[9]; unsigned char arg[9]; };
static const Kat KATS[4] = {
    {SeparableOperator::Top, {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 1, 0, 0, 0, 0, 0, 0, 0, 0, 4, 9, 5, 5, 11, 0, 0, 6, 9, 1},
     {0, 0, 0, 2, 0, 0, 9, 9, 11}, {3, 3, 3, 0, 3, 3, 1, 3, 0}},
    {SeparableOperator::Left, {0, 0, 0, 0, 0, 0, 0, 6, 7, 10, 0, 0, 4, 5, 10, 0, 0, 4, 6, 15, 0, 0, 1, 13, 21, 0, 0, 2, 15, 17},
     {0, 7, 10, 0, 6, 15, 0, 15, 21}, {3, 3, 2, 3, 3, 2, 3, 3, 0}},
    {SeparableOperator::Right, {0, 0, 0, 0, 0, 16, 12, 0, 0, 0, 14, 15, 0, 0, 0, 19, 24, 0, 0, 0, 22, 29, 0, 0, 0, 19, 27, 0, 0, 0},
     {16, 0, 0, 24, 0, 0, 29, 0, 0}, {2, 3, 3, 3, 3, 3, 1, 3, 3}},
    {SeparableOperator::Bottom, {0, 0, 0, 0, 0, 0, 0, 0, 1, 2, 0, 0, 4, 7, 8, 7, 20, 24, 20, 13, 0, 0, 0, 0, 0, 1, 1, 0, 0, 0},
     {0, 1, 2, 20, 24, 13, 1, 0, 0}, {3, 3, 2, 3, 2, 2, 3, 3, 3}},
};

static int run_gpu() {
    // kernel.rs:434-441: 30 x 30 ramp convolved with the identity kernel, SAME padding, is the ramp
    {
        std::vector<int> ramp(900);
        for (int i = 0; i < 900; ++i) ramp[i] = i;
        const DMatrix matrix = DMatrix::from_row_iterator(30, 30, ramp.begin());
        const DMatrix kernel = DMatrix::from_row_slice(3, 3, {0, 0, 0, 0, 1, 0, 0, 0, 0});
        EXPECT(matrix == matrix.convolve_2d(kernel, Padding::Same));
    }
    // Appendix B: separated SAME convolution (post-ReLU), pooling and its last-max-wins argmax, all four operators
    {
        const DMatrix x = DMatrix::from_row_iterator(6, 5, X65);
        for (const Kat& k : KATS) {
            const DMatrix conv = x.convolve_2d_separated(k.op, Padding::Same);
            EXPECT(conv == DMatrix::from_row_iterator(6, 5, k.conv));
            std::vector<uint8_t> arg;
            const DMatrix pooled = conv.pool_2d(Padding::Same, Pooling::Max, &arg);
            EXPECT(pooled == DMatrix::from_row_iterator(3, 3, k.pool));
            const DMatrix want_arg = DMatrix::from_row_iterator(3, 3, k.arg);   // row-major table -> column-major order
            bool same = arg.size() == 9;
            for (size_t i = 0; same && i < 9; ++i) same = arg[i] == static_cast<uint8_t>(want_arg.as_slice()[i]);
            EXPECT(same);
            EXPECT(conv.relu() == conv);                                         // already clamped (kernel.rs:206)
        }
    }
    // rcn.rs:530-538: weight_init -- a (100 -> 32) layer holds 32 * 100 weights
    {
        rcn::RCN model(10, {}, {32});
        model.init_params(100);
        EXPECT(model.layer_shape(0) == std::make_pair(size_t{32}, size_t{100}));
        EXPECT(model.layer_weights(0).m.len() == 32 * 100);
    }
    // Appendix B: one SGD step of the 3-2-2 sigmoid MLP (eta = 3, batch of one)
    {
        rcn::RCN model(2, {}, {2});
        model.init_params(3);
        model.set_weights(0, DMatrix::from_row_slice(2, 3, {0.1, -0.2, 0.3, 0.4, 0.5, -0.6}));
        model.set_bias(0, {0.01, -0.02});
        model.set_weights(1, DMatrix::from_row_slice(2, 2, {0.7, -0.8, -0.9, 1.0}));
        model.set_bias(1, {0.03, 0.04});
        const std::vector<double> a2 = model.classify_test({1.0, 0.5, -1.5});
        EXPECT(close(a2[0], 0.41256147606104177) && close(a2[1], 0.6246750573701205));
        model.train_batch({1.0, 0.5, -1.5}, {0.0, 1.0}, 1, 3.0);
        const DMatrix w2 = model.layer_weights(1).m, w1 = model.layer_weights(0).m;
        const double want_w2[4] = {0.5824940070747917, -1.046567695808136, -0.7965836352917443, 1.217002844877865};
        const double want_w1[6] = {-0.006645400939210289, -0.25332270046960514, 0.45996810140881544,
                                   0.47373513056408206, 0.536867565282041, -0.710602695846123};
        for (size_t r = 0; r < 2; ++r) {
            for (size_t c = 0; c < 2; ++c) EXPECT(close(w2(r, c), want_w2[r * 2 + c]));
            for (size_t c = 0; c < 3; ++c) EXPECT(close(w1(r, c), want_w1[r * 3 + c]));
        }
        const std::vector<double> b2 = model.layer_bias(1).v, b1 = model.layer_bias(0).v;
        EXPECT(close(b2[0], -0.26995839635852104) && close(b2[1], 0.3039917007029655));
        EXPECT(close(b1[0], -0.0966454009392103) && close(b1[1], 0.05373513056408204));
    }
    // RCN::train / classify on synthetic decoded sets: shapes, the log line, determinism under a fixed seed
    {
        auto make = [](size_t n, uint64_t seed) {
            rcn::GraySet s;
            s.n = n; s.h = 28; s.w = 28;
            s.pixels.resize(n * 784);
            s.labels.resize(n);
            std::mt19937_64 gen(seed);
            for (auto& p : s.pixels) p = static_cast<uint8_t>(gen() & 0xFF);
            for (size_t i = 0; i < n; ++i) s.labels[i] = static_cast<int64_t>(i % 10);
            return s;
        };
        const rcn::GraySet train = make(72, 1), test = make(30, 2);
        std::vector<uint64_t> first;
        std::vector<double> first_w;
        for (int rep = 0; rep < 2; ++rep) {
            rcn::RCN model(10, {rcn::RCNLayer::Convolve2D(Padding::Same), rcn::RCNLayer::Pool2D(Pooling::Max)}, {30}, "train", "test");
            std::ostringstream log;
            const std::vector<uint64_t> hist = model.train(train, test, 16, 2, 0.5, 7, &log);
            EXPECT(hist.size() == 2 && hist[0] <= 30 && hist[1] <= 30);
            EXPECT(model.layer_shape(0) == std::make_pair(size_t{30}, size_t{784}) && model.layer_shape(1) == std::make_pair(size_t{10}, size_t{30}));
            EXPECT(log.str().rfind("Epoch 0: ", 0) == 0 && log.str().find("/30 [") != std::string::npos);
            const std::vector<int64_t> labels = model.classify(test);
            EXPECT(labels.size() == 30);
            EXPECT(static_cast<int64_t>(model.classify(test.pixels.data(), 28, 28)) == labels[0]);
            const std::vector<double> w = model.layer_weights(0).m.as_slice();
            if (rep == 0) { first = hist; first_w = w; }
            else EXPECT(hist == first && w == first_w);          // same seed, same shuffles, same kernels: bit-identical
        }
    }
    if (!g_failed) std::printf("gpu ok\n");
    return g_failed ? 1 : 0;
}

int main(int argc, char** argv) {
    const std::string mode = argc > 1 ? argv[1] : "cpu";
    try {
        return mode == "gpu" ? run_gpu() : run_cpu(argc > 2 ? argv[2] : "/tmp");
    } catch (const std::exception& e) {
        std::printf("FAILED with exception: %s\n", e.what());
        return 2;
    }
}
