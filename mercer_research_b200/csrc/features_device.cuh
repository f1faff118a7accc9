// features_device.cuh -- device code of the feature stage (Sobel-separated conv, ReLU, 2x2 max-pool, flatten,
// standardise), shared by the stand-alone feature kernels (features.cu) and the fused training kernel (smallnet.cu).
// Reference: rcn/src/utils/kernel.rs:38-53,110-349; rcn/src/rcn.rs:41-46,317-356,407-412.
#pragma once
#include "features.cuh"

#include <cuda_fp16.h>

namespace rcn {

// ------------------------------------------------------------------------------------------------
// Device arithmetic.  mac(a, k, c) = c + a*k, the product rounded before the add like the reference's separate
// multiply and add (kernel.rs:164).  The taps are in {0, +-1, +-2}, so a*k is exact -- except that 2*a overflows for
// |a| > DBL_MAX / 2: the reference then adds +-Inf, where a fused multiply-add would round the exact sum to a finite
// value.  Zero taps are kept (inf*0 must stay NaN as in the reference); for T = int the compiler folds them away.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double mac(double a, double k, double c) { return __dadd_rn(c, __dmul_rn(a, k)); }
__device__ __forceinline__ int mac(int a, int k, int c) { return a * k + c; }

template <typename T>
__device__ __forceinline__ T relu1(T v) { return (v >= T(0)) ? v : T(0); }  // kernel.rs:214

// Pre-activation responses of the four operators (kernel.rs:38-53) at output pixel (y, x) of
// convolve_2d(3x1, p) . convolve_2d(1x3, p)  (kernel.rs:204-205), f is one h x w column-major map.
// SAME reproduces the reference's padded-copy quirk (kernel.rs:154-158, SURVEY.md A.2): the result is the
// Sobel response centred at (y-1, x-1); row 0 is zero; the last input column / last intermediate row are
// never read.
template <typename T, bool SAME>
__device__ __forceinline__ void sobel4(const T* __restrict__ f, int h, int w, int y, int x, T& t, T& l, T& r, T& b) {
    const T Z = T(0);
    T ct[3], cb[3], cs[3];  // vertical passes with [1,0,-1], [-1,0,1], [1,2,1] at the three columns
    if (SAME) {
        if (y == 0) { t = l = r = b = Z; return; }
        const int rr = y - 1;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int j = x + k - 2;
            if (j >= 0 && j <= w - 2) {
                const T* col = f + (size_t)j * h;
                const T x0 = (rr >= 1) ? col[rr - 1] : Z;
                const T x1 = col[rr];
                const T x2 = col[rr + 1];
                ct[k] = mac(x2, T(-1), mac(x1, T(0), mac(x0, T(1), Z)));
                cb[k] = mac(x2, T(1), mac(x1, T(0), mac(x0, T(-1), Z)));
                cs[k] = mac(x2, T(1), mac(x1, T(2), mac(x0, T(1), Z)));
            } else {
                ct[k] = cb[k] = cs[k] = Z;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const T* col = f + (size_t)(x + k) * h;
            const T x0 = col[y], x1 = col[y + 1], x2 = col[y + 2];
            ct[k] = mac(x2, T(-1), mac(x1, T(0), mac(x0, T(1), Z)));
            cb[k] = mac(x2, T(1), mac(x1, T(0), mac(x0, T(-1), Z)));
            cs[k] = mac(x2, T(1), mac(x1, T(2), mac(x0, T(1), Z)));
        }
    }
    t = mac(ct[2], T(1), mac(ct[1], T(2), mac(ct[0], T(1), Z)));   // Top:    h = [1,2,1]
    b = mac(cb[2], T(1), mac(cb[1], T(2), mac(cb[0], T(1), Z)));   // Bottom: h = [1,2,1]
    l = mac(cs[2], T(-1), mac(cs[1], T(0), mac(cs[0], T(1), Z)));  // Left:   h = [1,0,-1]
    r = mac(cs[2], T(1), mac(cs[1], T(0), mac(cs[0], T(-1), Z)));  // Right:  h = [-1,0,1]
}

template <typename T>
__device__ __forceinline__ void sobel4_relu(const Stage& st, const T* __restrict__ f, int y, int x, T& t, T& l, T& r, T& b) {
    if (st.same) sobel4<T, true>(f, st.h_in, st.w_in, y, x, t, l, r, b);
    else sobel4<T, false>(f, st.h_in, st.w_in, y, x, t, l, r, b);
    t = relu1(t); l = relu1(l); r = relu1(r); b = relu1(b);
}

// Iterator::max_by keeps the LAST maximal element (kernel.rs:278-281): replace unless strictly smaller.
template <typename T>
__device__ __forceinline__ void max_last(T& best, T v) { if (!(v < best)) best = v; }

// Exact-integer fast path for a Padding::Same conv directly followed by the 2x2 max-pool (the canonical rcn layer
// pair): the four conv pixels of one pooled output share a 4x4 input patch, the vertical passes are shared
// between Top/Bottom ([1,0,-1] and its negation) and Left/Right ([1,2,1]), and ReLU + max collapse to
// max(0, max T), max(0, -min T).  Integer arithmetic is exact, so this equals the literal tap chains of sobel4
// (and therefore the reference) bit for bit.
__device__ __forceinline__ void conv_pool_same_int(const int* __restrict__ f, int h, int w, int y, int x, int& t, int& l,
                                                   int& r, int& b) {
    int p[4][4];  // rows 2y-2 .. 2y+1, cols 2x-2 .. 2x+1
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = 2 * x - 2 + k;
        const bool cok = (c >= 0) && (c <= w - 2);  // intermediate columns outside [0, w-2] are zero (SURVEY.md A.2)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rr = 2 * y - 2 + i;
            p[i][k] = (cok && rr >= 0 && rr < h) ? f[c * h + rr] : 0;
        }
    }
    int tmax = 0, tmin = 0, lmax = 0, lmin = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int cy = 2 * y + a;
        const bool rok = (cy >= 1) && (cy < h);  // conv row 0 is zero; rows >= h are the pool's zero padding
        int vT[4], vS[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            vT[k] = p[a][k] - p[a + 2][k];
            vS[k] = p[a][k] + 2 * p[a + 1][k] + p[a + 2][k];
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool ok = rok && (2 * x + e < w);
            const int T = ok ? vT[e] + 2 * vT[e + 1] + vT[e + 2] : 0;
            const int L = ok ? vS[e] - vS[e + 2] : 0;
            tmax = max(tmax, T); tmin = min(tmin, T);
            lmax = max(lmax, L); lmin = min(lmin, L);
        }
    }
    t = tmax; b = -tmin; l = lmax; r = -lmin;
}

template <typename T>
__device__ __forceinline__ bool conv_pool_fast(const Stage&, const T*, int, int, T&, T&, T&, T&) { return false; }
template <>
__device__ __forceinline__ bool conv_pool_fast<int>(const Stage& st, const int* f, int y, int x, int& t, int& l, int& r, int& b) {
    if (!st.same) return false;
    conv_pool_same_int(f, st.h_in, st.w_in, y, x, t, l, r, b);
    return true;
}

// Runs one stage for one image.  `in`: n_in maps (column-major each, back to back).  emit(slot, y, x, v).
template <typename T, typename Emit>
__device__ __forceinline__ void run_stage(const Stage& st, const T* __restrict__ in, Emit emit, int tid, int nthreads) {
    const int hw_out = st.h_out * st.w_out;
    const int hw_in = st.h_in * st.w_in;
    const int items = st.n_in * hw_out;
    for (int it = tid; it < items; it += nthreads) {
        const int i = it / hw_out;
        const int rem = it - i * hw_out;
        const int x = rem / st.h_out;
        const int y = rem - x * st.h_out;
        const T* f = in + (size_t)i * hw_in;
        if (st.kind == 2) {
            // pool_2d(Padding::Same, Max): kernel.rs:245-349, zero row/col appended when odd.
            T best = T(0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int cy = 2 * y + (q >> 1), cx = 2 * x + (q & 1);
                const T v = (cy < st.h_in && cx < st.w_in) ? f[(size_t)cx * st.h_in + cy] : T(0);
                if (q == 0) best = v; else max_last(best, v);
            }
            emit(i, y, x, best);
            continue;
        }
        T t, l, r, b;
        if (st.kind == 0) {
            sobel4_relu<T>(st, f, y, x, t, l, r, b);
        } else if (!conv_pool_fast<T>(st, f, y, x, t, l, r, b)) {
            t = l = r = b = T(0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int cy = 2 * y + (q >> 1), cx = 2 * x + (q & 1);
                T vt = T(0), vl = T(0), vr = T(0), vb = T(0);
                if (cy < st.h_c && cx < st.w_c) sobel4_relu<T>(st, f, cy, cx, vt, vl, vr, vb);
                if (q == 0) { t = vt; l = vl; r = vr; b = vb; }
                else { max_last(t, vt); max_last(l, vl); max_last(r, vr); max_last(b, vb); }
            }
        }
        // Slot order (rcn.rs:325-339): first conv -> [T,L,R,B]; later convs overwrite slot i with Bottom and
        // append Top, Left, Right of map i at n + 3i.
        int sT, sL, sR, sB;
        if (st.first) { sT = 0; sL = 1; sR = 2; sB = 3; }
        else { sB = i; sT = st.n_in + 3 * i; sL = sT + 1; sR = sT + 2; }
        emit(sT, y, x, t); emit(sL, y, x, l); emit(sR, y, x, r); emit(sB, y, x, b);
    }
}

template <typename T>
struct EmitMaps {  // into a map set (shared or global), column-major maps back to back
    T* out; int h, hw;
    __device__ __forceinline__ void operator()(int slot, int y, int x, T v) const { out[(size_t)slot * hw + x * h + y] = v; }
};

template <typename T>
struct EmitFeatures {  // final stage: flatten (rcn.rs:350-355) + optional standardise/clamp (rcn.rs:407-412)
    double* out; int h, hw; Standardise sc;
    __device__ __forceinline__ void operator()(int slot, int y, int x, T v) const {
        double d = (double)v;
        if (sc.mode == 1) {
            d = (d - sc.mean) / sc.sd;                       // IEEE division
            d = (d >= 0.0) ? d : 0.0;
        } else if (sc.mode == 2) {
            // Markstein division: q = RN(a*r), rem = a - q*sd (exact in one fma), RN(q + rem*r) == RN(a/sd).
            // Only enabled after the host has checked bit-equality with IEEE division for EVERY value this
            // stage can produce with this (mean, sd) (standardise_fast_ok), so it is exact, not approximate.
            const double a = d - sc.mean;
            const double q = __dmul_rn(a, sc.rcp);
            const double rem = fma(-q, sc.sd, a);
            d = fma(rem, sc.rcp, q);
            d = (d >= 0.0) ? d : 0.0;
        }
        out[(size_t)slot * hw + x * h + y] = d;
    }
};

template <typename TIN, typename T>
__device__ __forceinline__ void load_image(const TIN* __restrict__ src, T* dst, int H, int W, int tid, int nthreads);

// u8 row-major (image crate) -> column-major T: DMatrix::from_row_iterator (lib.rs:29-33)
template <>
__device__ __forceinline__ void load_image<uint8_t, int>(const uint8_t* __restrict__ src, int* dst, int H, int W, int tid, int nthreads) {
    const int n = H * W;
    for (int i = tid; i < n; i += nthreads) { const int r = i / W, c = i - r * W; dst[c * H + r] = (int)src[i]; }
}
template <>
__device__ __forceinline__ void load_image<uint8_t, double>(const uint8_t* __restrict__ src, double* dst, int H, int W, int tid, int nthreads) {
    const int n = H * W;
    for (int i = tid; i < n; i += nthreads) { const int r = i / W, c = i - r * W; dst[c * H + r] = (double)src[i]; }
}
template <>
__device__ __forceinline__ void load_image<double, double>(const double* __restrict__ src, double* dst, int H, int W, int tid, int nthreads) {
    const int n = H * W;
    for (int i = tid; i < n; i += nthreads) dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------------
// Staged path (CpPlan, features.cuh): device side.
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int cp_pitch(int h) { return (h + 4) & ~1; }   // rows -2 .. h (+1 to stay even)
__host__ __device__ __forceinline__ int cp_cols(int w) { return w + 3; }            // cols -2 .. w
constexpr int kCpWordsPerTask = 4;

__device__ __forceinline__ int cp_div(int n, unsigned magic) { return (int)__umulhi((unsigned)n, magic); }   // divisor >= 2
__device__ __forceinline__ int cp_div1(int n, int d, unsigned magic) { return d == 1 ? n : cp_div(n, magic); }

namespace cpbulk {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk-async copy global -> shared, completion counted in bytes on `bar` (16-byte aligned, size % 16 == 0)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
}  // namespace cpbulk

// integer feature value -> f64 (exact: 0 <= v < 2^31) -> optional standardise + clamp (rcn.rs:407-412)
__device__ __forceinline__ double cp_finish(int mode, int v, const Standardise& sc) {
    double d = __hiloint2double(0x43300000, v) - 4503599627370496.0;   // (2^52 + v) - 2^52 == (double)v
    if (mode == 1) {
        d = (d - sc.mean) / sc.sd;
        d = (d >= 0.0) ? d : 0.0;
    } else if (mode == 2) {   // host-verified exact Markstein division, see EmitFeatures
        const double a = d - sc.mean;
        const double q = __dmul_rn(a, sc.rcp);
        const double rem = fma(-q, sc.sd, a);
        d = fma(rem, sc.rcp, q);
        d = (d >= 0.0) ? d : 0.0;
    }
    return d;
}

template <int MODE>
struct CpSinkGlobal {   // flattened feature vector of one image in global memory (rcn.rs:350-355)
    double* gout; Standardise sc;
    __device__ __forceinline__ void operator()(int idx, int v) const { gout[idx] = cp_finish(MODE, v, sc); }
};

// One pooled output position of a conv(Same)+pool stage over padded int32 tiles: item `it` of one image =
// (map i, column x, row y), y fastest.  LAST: the four operator responses go to `sink(feature index, value)`; otherwise
// into the next stage's padded tiles `nxt` (whose last column stays zero).  Exact int32 closed form of
// conv_pool_same_int without a single bounds test on the loads.
template <bool LAST, bool FIRST, typename Sink>
__device__ __forceinline__ void cp_item(const CpStage& st, const int* __restrict__ in, int it, int* __restrict__ nxt,
                                        int nxt_hp, int nxt_map, const Sink& sink) {
    const int hw_out = st.h_out * st.w_out;
    const int hp = st.hp;
    int i = 0, rem = it;
    if (!FIRST) { i = cp_div(it, st.magic_hw); rem = it - i * hw_out; }
    const int x = cp_div(rem, st.magic_h);
    const int y = rem - x * st.h_out;
    // padded coordinates: image (row r, col c) sits at [(c + 2) * hp + r + 2]; the patch starts at (2y-2, 2x-2)
    const int* f = in + i * st.map_elems + (2 * x) * hp + 2 * y;
    int p[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int2 a = *reinterpret_cast<const int2*>(f + k * hp);
        const int2 b = *reinterpret_cast<const int2*>(f + k * hp + 2);
        p[0][k] = a.x; p[1][k] = a.y; p[2][k] = b.x; p[3][k] = b.y;
    }
    // conv row 2y+a is zero for row 0 (SURVEY.md A.2) and beyond the map (the pool's zero padding, kernel.rs:253-261)
    const bool rok0 = y > 0, rok1 = 2 * y + 1 < st.h;
    const bool cok1 = 2 * x + 1 < st.w;
    int tmax = 0, tmin = 0, lmax = 0, lmin = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        int vT[4], vS[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            vT[k] = p[a][k] - p[a + 2][k];
            vS[k] = p[a][k] + 2 * p[a + 1][k] + p[a + 2][k];
        }
        const bool rok = a ? rok1 : rok0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool ok = rok && (e ? cok1 : true);
            const int T = ok ? vT[e] + 2 * vT[e + 1] + vT[e + 2] : 0;
            const int L = ok ? vS[e] - vS[e + 2] : 0;
            tmax = max(tmax, T); tmin = min(tmin, T);
            lmax = max(lmax, L); lmin = min(lmin, L);
        }
    }
    const int t = tmax, b = -tmin, l = lmax, r = -lmin;
    // slot order rcn.rs:325-339: first conv [T,L,R,B]; later convs put Bottom in slot i and T,L,R at n + 3i
    const int sB = FIRST ? 3 : i;
    const int sT = FIRST ? 0 : st.n_in + 3 * i;
    if (LAST) {
        const int o = sT * hw_out + rem;                  // rem == x * h_out + y
        sink(o, t);
        sink(o + hw_out, l);
        sink(o + 2 * hw_out, r);
        sink(sB * hw_out + rem, b);
    } else if (x < st.w_out - 1) {
        int* o = nxt + sT * nxt_map + (x + 2) * nxt_hp + y + 2;
        o[0] = t;
        o[nxt_map] = l;
        o[2 * nxt_map] = r;
        nxt[sB * nxt_map + (x + 2) * nxt_hp + y + 2] = b;
    }
}

// ------------------------------------------------------------------------------------------------
// Packed form of a ONE-stage plan: the two fp16 lanes of a tile word hold the same pixel of two images.  From u8 pixels, every
// intermediate of the closed form above is an integer of magnitude <= 255 * 4 = 1020 and fp16 holds every integer up to 2048
// exactly, so HADD2 / HFMA2 (tap 2) / HMNMX2 compute both images' values exactly, one instruction for the pair.  (A second
// stage would reach 255 * 16: more stages keep the int32 tiles.)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ __half2 cp_h2(uint32_t u) { return *reinterpret_cast<const __half2*>(&u); }
__device__ __forceinline__ uint32_t cp_u32(__half2 h) { return *reinterpret_cast<const uint32_t*>(&h); }

// cp_item<true, true> over packed tiles: the four features of the pair's image in lane .x go to sink_x, those of lane .y to
// sink_y (skipped when `live_y` is false: that lane is a zero image).
template <typename Sink>
__device__ __forceinline__ void cp_item_pair(const CpStage& st, const uint32_t* __restrict__ in, int it, const Sink& sink_x,
                                             const Sink& sink_y, bool live_y) {
    const int hw_out = st.h_out * st.w_out;
    const int hp = st.hp;
    const int x = cp_div(it, st.magic_h);
    const int y = it - x * st.h_out;
    const uint32_t* f = in + (2 * x) * hp + 2 * y;
    __half2 p[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint2 a = *reinterpret_cast<const uint2*>(f + k * hp);
        const uint2 b = *reinterpret_cast<const uint2*>(f + k * hp + 2);
        p[0][k] = cp_h2(a.x); p[1][k] = cp_h2(a.y); p[2][k] = cp_h2(b.x); p[3][k] = cp_h2(b.y);
    }
    const bool rok0 = y > 0, rok1 = 2 * y + 1 < st.h;
    const bool cok1 = 2 * x + 1 < st.w;
    const __half2 zero = __float2half2_rn(0.0f), two = __float2half2_rn(2.0f);
    __half2 tmax = zero, tmin = zero, lmax = zero, lmin = zero;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        __half2 vT[4], vS[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            vT[k] = __hsub2(p[a][k], p[a + 2][k]);
            vS[k] = __hfma2(two, p[a + 1][k], __hadd2(p[a][k], p[a + 2][k]));
        }
        const bool rok = a ? rok1 : rok0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool ok = rok && (e ? cok1 : true);
            const __half2 T = ok ? __hfma2(two, vT[e + 1], __hadd2(vT[e], vT[e + 2])) : zero;
            const __half2 L = ok ? __hsub2(vS[e], vS[e + 2]) : zero;
            tmax = __hmax2(tmax, T); tmin = __hmin2(tmin, T);
            lmax = __hmax2(lmax, L); lmin = __hmin2(lmin, L);
        }
    }
    // t = tmax, b = -tmin, l = lmax, r = -lmin, each in [0, 1020]: 1024 + v is exact and its fp16 mantissa field is v
    const __half2 k1024 = __float2half2_rn(1024.0f);
    const uint32_t t = cp_u32(__hadd2(k1024, tmax)), b = cp_u32(__hsub2(k1024, tmin));
    const uint32_t l = cp_u32(__hadd2(k1024, lmax)), r = cp_u32(__hsub2(k1024, lmin));
    sink_x(it, (int)(t & 0x3FF));
    sink_x(it + hw_out, (int)(l & 0x3FF));
    sink_x(it + 2 * hw_out, (int)(r & 0x3FF));
    sink_x(it + 3 * hw_out, (int)(b & 0x3FF));
    if (live_y) {
        sink_y(it, (int)((t >> 16) & 0x3FF));
        sink_y(it + hw_out, (int)((l >> 16) & 0x3FF));
        sink_y(it + 2 * hw_out, (int)((r >> 16) & 0x3FF));
        sink_y(it + 3 * hw_out, (int)((b >> 16) & 0x3FF));
    }
}

// u8 row-major staging buffers -> packed fp16 tiles of a one-stage plan for n_img images: pair q holds image q in lane .x and
// image q + y_off in lane .y (staging at stg + image * stg_stride bytes, tiles at tiles + q * tile_stride words); lanes of images
// >= n_img are zero.  Byte k of both images' words is placed in the low byte of each half by one byte permute, given the
// exponent of 1024 (0x6400: the half 1024 + byte, exact) and shifted back by 1024 with one HSUB2.  Task geometry and bank
// pattern as cp_transpose_images below, over the pairs.
__device__ __forceinline__ void cp_transpose_pairs(const uint8_t* __restrict__ stg, int stg_stride, int y_off,
                                                   uint32_t* __restrict__ tiles, int tile_stride, int n_img, int H, int W,
                                                   const CpPlan& cp, int tid, int nt) {
    const int W4 = W >> 2;
    const int hp = cp.s[0].hp;
    const int chunks = (W4 + kCpWordsPerTask - 1) / kCpWordsPerTask;
    const int tpi = cp.tasks_per_image;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    const int n_pairs = min(y_off, n_img);
    const __half2 k1024 = __float2half2_rn(1024.0f);
    for (int task = warp; task < n_pairs * tpi; task += nwarps) {
        const int q = cp_div1(task, tpi, cp.magic_tasks);
        const int tl = task - q * tpi;
        const int rg = cp_div1(tl, chunks, cp.magic_chunks);
        const int it0 = (tl - rg * chunks) * kCpWordsPerTask;
        const int r = rg * 32 + lane;
        if (r >= H) continue;
        int j = lane + it0;
        if (W4 > 1) j -= cp_div(j, cp.magic_w4) * W4; else j = 0;
        const uint32_t* row_x = reinterpret_cast<const uint32_t*>(stg + (size_t)q * stg_stride) + r * W4;
        const uint32_t* row_y = reinterpret_cast<const uint32_t*>(stg + (size_t)(q + y_off) * stg_stride) + r * W4;
        const bool live_y = q + y_off < n_img;
        uint32_t* col0 = tiles + q * tile_stride + 2 * hp + r + 2;
        const int n = min(kCpWordsPerTask, W4 - it0);
#pragma unroll
        for (int u = 0; u < kCpWordsPerTask; ++u) {
            if (u < n) {
                const uint32_t vx = row_x[j];
                const uint32_t vy = live_y ? row_y[j] : 0u;
                uint32_t* dst = col0 + 4 * j * hp;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (k == 3 && j == W4 - 1) break;   // column W-1 is never read downstream and stays zero
                    // selector nibble n picks result byte n: byte k of vx -> byte 0, byte k of vy (index 4 + k) -> byte 2
                    const uint32_t w = (__byte_perm(vx, vy, (unsigned)(k | ((k + 4) << 8))) & 0x00FF00FFu) | 0x64006400u;
                    dst[k * hp] = cp_u32(__hsub2(cp_h2(w), k1024));
                }
                j = (j + 1 == W4) ? 0 : j + 1;
            }
        }
    }
}

// u8 row-major staging buffers -> padded int32 column-major tiles of stage 0 (lib.rs:29-33 layout change) for G images
// (image g: staging at stg + g*stg_stride bytes, tiles at tiles + g*tile_stride ints).  Lane l of a warp task takes
// row r0 + l and walks words (l + it) mod W/4 of that row: the 4-byte reads and the four column-strided writes are both
// bank-conflict free.  Column W-1 is never read downstream and stays zero.
__device__ __forceinline__ void cp_transpose_images(const uint8_t* __restrict__ stg, int stg_stride, int* __restrict__ tiles,
                                                    int tile_stride, int G, int H, int W, const CpPlan& cp, int tid, int nt) {
    const int W4 = W >> 2;
    const int hp = cp.s[0].hp;
    const int chunks = (W4 + kCpWordsPerTask - 1) / kCpWordsPerTask;
    const int tpi = cp.tasks_per_image;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    for (int task = warp; task < G * tpi; task += nwarps) {
        const int g = cp_div1(task, tpi, cp.magic_tasks);
        const int tl = task - g * tpi;
        const int rg = cp_div1(tl, chunks, cp.magic_chunks);
        const int it0 = (tl - rg * chunks) * kCpWordsPerTask;
        const int r = rg * 32 + lane;
        if (r >= H) continue;
        int j = lane + it0;
        if (W4 > 1) j -= cp_div(j, cp.magic_w4) * W4; else j = 0;
        const uint32_t* row = reinterpret_cast<const uint32_t*>(stg + (size_t)g * stg_stride) + r * W4;
        int* col0 = tiles + g * tile_stride + 2 * hp + r + 2;
        const int n = min(kCpWordsPerTask, W4 - it0);
#pragma unroll
        for (int u = 0; u < kCpWordsPerTask; ++u) {
            if (u < n) {
                const uint32_t v = row[j];
                int* dst = col0 + 4 * j * hp;
                dst[0] = (int)__byte_perm(v, 0, 0x4440);
                dst[hp] = (int)__byte_perm(v, 0, 0x4441);
                dst[2 * hp] = (int)__byte_perm(v, 0, 0x4442);
                if (j != W4 - 1) dst[3 * hp] = (int)__byte_perm(v, 0, 0x4443);
                j = (j + 1 == W4) ? 0 : j + 1;
            }
        }
    }
}

__device__ __forceinline__ size_t source_image(const BatchIndex& bi, size_t img) {
    if (!bi.cursor) return img;
    const long long pos = __ldcg(bi.cursor) + (long long)img;   // L2: a persistent kernel advances the cursor between steps
    return (size_t)(bi.perm ? bi.perm[pos] : pos);
}
// Streamed epoch, copy-engine mode: block until image `src` of the walk has landed in the ring (BatchIndex::arrived).  The
// counter is written by the copy stream right behind the copy that carried the image, so an acquire load that sees it also
// orders the image bytes; the proxy fence extends that to the bulk-async loads issued next.  A copy that has not arrived after
// 20 s is a broken copy stream: trap (the host call then fails with the CUDA error instead of training on garbage).
__device__ __forceinline__ void wait_arrived(const BatchIndex& bi, size_t src) {
    if (!bi.arrived) return;
    long long a;
    asm volatile("ld.acquire.sys.global.s64 %0, [%1];" : "=l"(a) : "l"(bi.arrived) : "memory");
    if (a <= (long long)src) {
        unsigned long long t0, t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        do {
            __nanosleep(200);
            asm volatile("ld.acquire.sys.global.s64 %0, [%1];" : "=l"(a) : "l"(bi.arrived) : "memory");
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > 20000000000ull) __trap();
        } while (a <= (long long)src);
    }
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
// where that image's pixels live: the dataset itself, or a ring of `window` slots when streaming from the host
__device__ __forceinline__ size_t image_slot(const BatchIndex& bi, size_t src) {
    return bi.window ? (size_t)((unsigned)src % (unsigned)bi.window) : src;   // 32-bit: a streamed epoch has < 2^32 samples
}


}  // namespace rcn
