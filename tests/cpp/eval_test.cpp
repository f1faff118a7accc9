// rcn::RCN::evaluate_images through the C++ mirror (include/rcn.hpp).
//   eval_test cpu   the devices are hidden: constructing a model throws rcn::Error with RCN_ERR_CUDA (no CPU fallback)
//   eval_test gpu   on cuda:0, evaluate_images agrees with the exact-one-hot hit rule and the quadratic cost computed on the
//                   host from the library's features + forward pass (rcn_cuda_features, rcn_cuda_forward), ties included
#include "rcn.hpp"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>

static int fail(const char* what) {
    std::printf("FAIL: %s\n", what);
    return 1;
}

static rcn::RCN canonical() {
    return rcn::RCN(10, {rcn::RCNLayer::Convolve2D(rcn::Padding::Same), rcn::RCNLayer::Pool2D(rcn::Pooling::Max)}, {30});
}

int main(int argc, char** argv) {
    if (argc < 2) return fail("usage: eval_test cpu|gpu");
    const std::string mode = argv[1];
    if (mode == "cpu") {
        try {
            rcn::RCN m = canonical();
            return fail("a CUDA device is present");
        } catch (const rcn::Error& e) {
            if (e.status != RCN_ERR_CUDA) return fail("expected RCN_ERR_CUDA");
        }
        std::printf("cpu ok\n");
        return 0;
    }
    if (mode != "gpu") return fail("unknown mode");
    rcn::RCN m = canonical();
    m.load_weights_and_bias(m.feature_len(28, 28), 42);
    m.set_scale_set({40.0, 60.0});
    {   // outputs 0 and 1 get the same weights and bias: they are always equal, so a sample whose maximum is there has a tied
        // maximum and is never a hit, even with label 0 or 1 (a plain argmax comparison would count label 1 as one)
        rcn::Weights w = m.layer_weights(1);
        double* p = w.m.as_mut_ptr();
        for (size_t c = 0; c < w.m.ncols(); ++c) p[c * w.m.nrows() + 1] = p[c * w.m.nrows()];
        m.set_weights(1, w.m);
        rcn::Bias b = m.layer_bias(1);
        b.v[1] = b.v[0];
        m.set_bias(1, b.v);
    }
    rcn::GraySet set;
    set.n = 500; set.h = 28; set.w = 28;
    std::mt19937_64 gen(7);
    set.pixels.resize(set.n * 28 * 28);
    for (uint8_t& p : set.pixels) p = static_cast<uint8_t>(gen() & 255);
    const std::vector<int64_t> pred = m.classify(set);
    set.labels.resize(set.n);
    for (size_t i = 0; i < set.n; ++i) set.labels[i] = (i % 2) ? static_cast<int64_t>(gen() % 10) : pred[i];
    // the host side of rcn.rs:152-157 on the library's forward pass: hit iff {i : a_i == max a} == {label}; cost 0.5 |a - y|^2
    const size_t L = m.feature_len(28, 28), C = 10;
    std::vector<double> feats(L * set.n), acts(C * set.n);
    rcn::check(rcn_cuda_features(m.handle(), set.pixels.data(), RCN_PIXELS_U8_ROWMAJOR, set.n, 28, 28, 1, feats.data()));
    rcn::check(rcn_cuda_forward(m.handle(), feats.data(), set.n, acts.data()));
    uint64_t want = 0, ties = 0;
    double want_cost = 0.0;
    for (size_t b = 0; b < set.n; ++b) {
        const double* a = &acts[b * C];
        double mx = a[0];
        for (size_t i = 1; i < C; ++i) mx = std::fmax(mx, a[i]);
        bool ok = true;
        size_t n_max = 0;
        for (size_t i = 0; i < C; ++i) {
            const double y = set.labels[b] == (int64_t)i ? 1.0 : 0.0;
            want_cost += 0.5 * (a[i] - y) * (a[i] - y);
            ok = ok && ((a[i] == mx ? 1.0 : 0.0) == y);
            n_max += a[i] == mx;
        }
        want += ok;
        ties += n_max > 1;
    }
    const auto [accept, cost] = m.evaluate_images(set);
    if (accept != want) {
        std::printf("accept %llu, host rule says %llu\n", (unsigned long long)accept, (unsigned long long)want);
        return fail("accept count");
    }
    if (!(std::fabs(cost - want_cost) <= 1e-9 * std::fabs(want_cost))) {
        std::printf("cost %.17g, host sum %.17g\n", cost, want_cost);
        return fail("cost");
    }
    if (ties == 0) return fail("no sample with tied outputs: the exact-one-hot rule was not exercised");
    rcn::GraySet empty;
    empty.h = 28; empty.w = 28;
    if (m.evaluate_images(empty) != std::make_pair<uint64_t, double>(0, 0.0)) return fail("empty set");
    std::printf("accept %llu / %zu (%llu with tied outputs), cost %.6f\ngpu ok\n", (unsigned long long)accept, set.n,
                (unsigned long long)ties, cost);
    return 0;
}
