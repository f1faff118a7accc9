// ozaki.cu -- operand slicing and TMA descriptors for the tcgen05 integer-slice GEMM (see ozaki.cuh for the scheme).
//
// Slicing is HBM-bound byte work (8 B read, 6 B written per element, twice over the operand because the per-row scale
// needs the row maximum first; the second sweep is served by L2 for the row blocks a CTA owns): coalesced loads along
// the operand's contiguous dimension, and for operands whose contraction index is NOT the contiguous one a
// shared-memory tile transpose so that the int8 planes are always written k-contiguous in 64-byte runs.
#include "ozaki.cuh"

#include <cuda_runtime_api.h>

namespace rcn {

namespace {

// x = scale * (q_0 + sum_{j>=1} d_j 2^(-8j)) with BALANCED digits: t = x * 2^(6-e) in (-64, 64); q_0 = rint(t);
// r = t - q_0 in [-0.5, 0.5]; d_j = rint(256 r), r = 256 r - d_j ...  Every step is exact in f64.  A digit that rounds
// to +128 (r within 2^-9 of +0.5) is rewritten as -128 with a carry into the next more significant digit, so all
// planes are int8 with zero-mean digits (dropped terms then add up like sqrt(K), not K); |q_0| <= 65.
__device__ __forceinline__ void slice6(double x, double inv, int8_t (&q)[OZ_S]) {
    int d[OZ_S];
    double t = x * inv;
    double f = rint(t);
    d[0] = (int)f;
    t = (t - f) * 256.0;
#pragma unroll
    for (int j = 1; j < OZ_S; ++j) {
        f = rint(t);
        d[j] = (int)f;
        t = (t - f) * 256.0;
    }
#pragma unroll
    for (int j = OZ_S - 1; j >= 1; --j) {
        const int carry = d[j] == 128 ? 1 : 0;
        d[j] -= carry << 8;
        d[j - 1] += carry;
    }
#pragma unroll
    for (int j = 0; j < OZ_S; ++j) q[j] = (int8_t)d[j];
}

// row scale from the row maximum: amax = f * 2^e, f in [0.5, 1)  =>  |x| * 2^-e < 1
// A row that holds a NaN / Inf (amax arrives as NaN, see amax_fold) or a magnitude the digit scaling cannot represent gets
// all-zero planes and scale = NaN: the epilogue's `acc * scale_a * scale_b` then yields NaN for every output that row
// touches, like the f64 DMMA / SIMT paths and the reference (NaN * x = NaN), instead of a silently finite result.
__device__ __forceinline__ void row_scale(double amax, double& inv, double& scale) {
    if (!(amax < 1e290)) { inv = 0.0; scale = __longlong_as_double(0x7FF8000000000000ll); return; }   // NaN / Inf / overflow-range row
    if (!(amax > 1e-290)) { inv = 0.0; scale = 0.0; return; }                                          // zero / denormal row: all-zero planes
    int e;
    frexp(amax, &e);
    inv = ldexp(1.0, 6 - e);
    scale = ldexp(1.0, e - 6);
}

// Row-maximum accumulation that does not lose non-finite values: fmax() drops NaN operands, so a NaN or Inf element turns
// the running maximum into +Inf (sticky under fmax); amax_finish() maps that to NaN for row_scale.
__device__ __forceinline__ double amax_fold(double amax, double v) {
    const double a = fabs(v);
    return (a <= 1.7976931348623157e308) ? fmax(amax, a) : __longlong_as_double(0x7FF0000000000000ll);
}
__device__ __forceinline__ double amax_finish(double amax) {
    return (amax <= 1.7976931348623157e308) ? amax : __longlong_as_double(0x7FF8000000000000ll);
}

// One row of a k-contiguous operand: a strided matrix row, or the im2col row of one grid pixel (gathered, zero padded).
struct RowReader {
    const double* row;      // dense
    ConvGeom g;             // gather
    int base, oy, ox;       // b*Hi*Wi, oy - ph, ox - pw
    bool gather;
    __device__ __forceinline__ RowReader(const OzOperand& op, int r) : row(nullptr), g(op.g), base(0), oy(0), ox(0), gather(op.gather == 1) {
        if (!gather) { row = op.p + (size_t)r * op.ld; return; }
        const int n = r + op.pix0;
        const int b = n / (g.Ho * g.Wo);
        const int rem = n - b * g.Ho * g.Wo;
        oy = rem / g.Wo;
        ox = rem - oy * g.Wo - g.pw;
        oy -= g.ph;
        base = b * g.Hi * g.Wi;
    }
    __device__ __forceinline__ double at(int k) const {
        if (!gather) return row[k];
        const int tap = k / g.C, c = k - tap * g.C;
        const int ky = tap / g.kw, kx = tap - ky * g.kw;
        const int iy = oy + ky, ix = ox + kx;
        if ((unsigned)iy >= (unsigned)g.Hi || (unsigned)ix >= (unsigned)g.Wi) return 0.0;
        return g.t[((size_t)(base + iy * g.Wi + ix)) * g.C + c];
    }
};

// k-contiguous operand: one warp per row.
__global__ void __launch_bounds__(256) ozaki_slice_kmajor_kernel(const OzOperand op, int R, int K, int Kp,
                                                                 int8_t* __restrict__ planes, double* __restrict__ scale) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + warp;
    if (r >= R) return;
    const RowReader row(op, r);
    double amax = 0.0;
    for (int k = lane; k < K; k += 32) amax = amax_fold(amax, row.at(k));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));   // +Inf marks a non-finite element
    double inv, sc;
    row_scale(amax_finish(amax), inv, sc);
    if (lane == 0) scale[r] = sc;
    const size_t plane = (size_t)R * Kp;
    for (int k4 = lane * 4; k4 < Kp; k4 += 128) {
        int8_t q[4][OZ_S];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k4 + u;
            slice6(k < K ? row.at(k) : 0.0, inv, q[u]);
        }
#pragma unroll
        for (int j = 0; j < OZ_S; ++j) {
            const uint32_t w = (uint32_t)(uint8_t)q[0][j] | ((uint32_t)(uint8_t)q[1][j] << 8) | ((uint32_t)(uint8_t)q[2][j] << 16) |
                               ((uint32_t)(uint8_t)q[3][j] << 24);
            *reinterpret_cast<uint32_t*>(planes + (size_t)j * plane + (size_t)r * Kp + k4) = w;
        }
    }
}

// element (r, k) at X[k*ld + r] (r contiguous).  Two kernels so that the machine is full even for 4096-row operands:
//   amax:  grid (rows/32, k-splits), per-row maxima combined with atomicMax on the bit pattern (|x| >= 0: bit order ==
//          value order), 8 loads in flight per thread;
//   slice: grid (rows/32, k-chunks of RM_KCHUNK): slices a 32-row x 64-k tile at a time and transposes it through
//          shared memory so the int8 planes are written k-contiguous in 64-byte runs.
constexpr int TR_PITCH = 68;   // bytes per (slice, row) line of the 64-k tile: 17 words -> conflict-free byte scatter
constexpr int RM_KCHUNK = 512;

// One row-contiguous operand column r seen along k: a strided matrix, or im2col column (ky, kx, c) over grid pixels.
struct ColReader {
    const double* p; size_t ld;   // dense
    ConvGeom g; int dy, dx, c, pix0;
    bool gather, valid;
    __device__ __forceinline__ ColReader(const OzOperand& op, int r, int R)
        : p(op.p), ld(op.ld), g(op.g), dy(0), dx(0), c(0), pix0(op.pix0), gather(op.gather == 2), valid(r < R) {
        if (!gather) { p = op.p + r; return; }
        if (!valid) return;
        const int tap = r / g.C;
        c = r - tap * g.C;
        const int ky = tap / g.kw;
        dy = ky - g.ph;
        dx = (tap - ky * g.kw) - g.pw;
    }
    __device__ __forceinline__ double at(int k) const {
        if (!gather) return p[(size_t)k * ld];
        const int pix = k + pix0;
        const int b = pix / (g.Ho * g.Wo);
        const int rem = pix - b * g.Ho * g.Wo;
        const int oy = rem / g.Wo, ox = rem - oy * g.Wo;
        const int iy = oy + dy, ix = ox + dx;
        if ((unsigned)iy >= (unsigned)g.Hi || (unsigned)ix >= (unsigned)g.Wi) return 0.0;
        return g.t[((size_t)((b * g.Hi + iy) * g.Wi + ix)) * g.C + c];
    }
};

__global__ void __launch_bounds__(256) ozaki_amax_rmajor_kernel(const OzOperand op, int R, int K, int k_per_cta,
                                                                unsigned long long* __restrict__ amax_bits) {
    __shared__ double red[8][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * 32 + lane;
    const int k_lo = blockIdx.y * k_per_cta, k_hi = min(K, k_lo + k_per_cta);
    const ColReader col(op, r, R);
    double amax = 0.0;
    if (r < R) {
        for (int k = k_lo + warp; k < k_hi; k += 64) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (k + 8 * u < k_hi) ? col.at(k + 8 * u) : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) amax = amax_fold(amax, v[u]);
        }
    }
    red[warp][lane] = amax;
    __syncthreads();
    if (warp == 0 && r < R) {
#pragma unroll
        for (int w = 1; w < 8; ++w) amax = fmax(amax, red[w][lane]);   // +Inf (a non-finite element) is sticky
        // bit order == value order for |x| >= 0; the quiet-NaN pattern sorts above +Inf, so it poisons the row for good
        atomicMax(amax_bits + r, (unsigned long long)__double_as_longlong(amax_finish(amax)));
    }
}

__global__ void __launch_bounds__(256) ozaki_slice_rmajor_kernel(const OzOperand op, int R, int K, int Kp,
                                                                 const unsigned long long* __restrict__ amax_bits,
                                                                 int8_t* __restrict__ planes, double* __restrict__ scale) {
    __shared__ double s_inv[32];
    __shared__ __align__(4) int8_t tile[OZ_S][32][TR_PITCH];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r0 = blockIdx.x * 32;
    const int r = r0 + lane;
    const bool rok = r < R;
    if (warp == 0) {
        double inv = 0.0, sc = 0.0;
        // im2col columns (ky, kx, c): the maximum over the pixels is the channel's maximum for every tap (an upper bound at
        // the borders), so one per-CHANNEL maximum serves all kh*kw rows of that channel
        if (rok) row_scale(__longlong_as_double((long long)amax_bits[op.gather == 2 ? r % op.g.C : r]), inv, sc);
        s_inv[lane] = inv;
        if (rok && blockIdx.y == 0) scale[r] = sc;
    }
    __syncthreads();
    const double inv = s_inv[lane];
    const ColReader col(op, r, R);
    const size_t plane = (size_t)R * Kp;
    const int kb_lo = blockIdx.y * RM_KCHUNK, kb_hi = min(Kp, kb_lo + RM_KCHUNK);
    for (int kb = kb_lo; kb < kb_hi; kb += 64) {
        double v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = kb + warp * 8 + j;
            v[j] = (rok && k < K) ? col.at(k) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int8_t q[OZ_S];
            slice6(v[j], inv, q);
#pragma unroll
            for (int s = 0; s < OZ_S; ++s) tile[s][lane][warp * 8 + j] = q[s];
        }
        __syncthreads();
        // write-out: per (slice, row) 64 contiguous bytes = 16 words
#pragma unroll
        for (int i = 0; i < OZ_S * 32 * 16 / 256; ++i) {
            const int idx = threadIdx.x + i * 256;
            const int s = idx / 512, rem = idx % 512;
            const int rr = rem / 16, w = rem % 16;
            if (r0 + rr < R)
                *reinterpret_cast<uint32_t*>(planes + (size_t)s * plane + (size_t)(r0 + rr) * Kp + kb + 4 * w) =
                    *reinterpret_cast<const uint32_t*>(&tile[s][rr][4 * w]);
        }
        __syncthreads();
    }
}

// ---- per-image slicing (one scale per image): convolution inputs whose im2col is done by TMA -----------------------
// x is [B][per_img]; blockIdx.y strides over the images, so a warp's maximum never mixes two images.  One scale per image
// keeps every output's truncation relative to its own image (a 128-pixel tile never crosses an image, see
// ozaki_conv_tma_ok), and a non-finite element poisons only its own image.
__global__ void __launch_bounds__(256) ozaki_amax_tensor_kernel(const double* __restrict__ x, int B, size_t per_img,
                                                                unsigned long long* __restrict__ amax_bits) {
    for (int img = blockIdx.y; img < B; img += gridDim.y) {
        const double* xi = x + (size_t)img * per_img;
        double amax = 0.0;
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per_img; i += (size_t)gridDim.x * blockDim.x)
            amax = amax_fold(amax, xi[i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        if ((threadIdx.x & 31) == 0) atomicMax(amax_bits + img, (unsigned long long)__double_as_longlong(amax_finish(amax)));
    }
}

__global__ void __launch_bounds__(256) ozaki_slice_tensor_kernel(const double* __restrict__ x, int B, size_t per_img,
                                                                 const unsigned long long* __restrict__ amax_bits,
                                                                 int8_t* __restrict__ planes, double* __restrict__ scale_out) {
    const size_t n = (size_t)B * per_img;
    const size_t n4 = per_img / 4;   // per_img is a multiple of 64 (C % 64 == 0)
    for (int img = blockIdx.y; img < B; img += gridDim.y) {
        double inv, sc;
        row_scale(__longlong_as_double((long long)amax_bits[img]), inv, sc);
        if (blockIdx.x == 0 && threadIdx.x == 0) scale_out[img] = sc;
        const double2* xi = reinterpret_cast<const double2*>(x + (size_t)img * per_img);
        uint32_t* pi = reinterpret_cast<uint32_t*>(planes + (size_t)img * per_img);
        for (size_t i4 = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i4 < n4; i4 += (size_t)gridDim.x * blockDim.x) {
            const double2 a = xi[2 * i4], b = xi[2 * i4 + 1];
            int8_t q[4][OZ_S];
            slice6(a.x, inv, q[0]); slice6(a.y, inv, q[1]); slice6(b.x, inv, q[2]); slice6(b.y, inv, q[3]);
#pragma unroll
            for (int j = 0; j < OZ_S; ++j) {
                const uint32_t w = (uint32_t)(uint8_t)q[0][j] | ((uint32_t)(uint8_t)q[1][j] << 8) | ((uint32_t)(uint8_t)q[2][j] << 16) |
                                   ((uint32_t)(uint8_t)q[3][j] << 24);
                pi[(size_t)j * (n / 4) + i4] = w;
            }
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

}  // namespace

bool ozaki_available() { return encode_tiled_fn() != nullptr; }

int ozaki_slice(const OzOperand& op, int rows, int K, int Kp, int8_t* planes, double* scale, double* scale_scratch,
                cudaStream_t stream) {
    if (rows <= 0) return RCN_OK;
    if (op.kcontig) {
        RCN_LAUNCH("ozaki_slice_kmajor_kernel", stream,
                   ozaki_slice_kmajor_kernel<<<cdiv(rows, 8), 256, 0, stream>>>(op, rows, K, Kp, planes, scale));
    } else {
        // the scale array doubles as the per-row |x| maximum (bit pattern) between the two kernels
        unsigned long long* amax_bits = reinterpret_cast<unsigned long long*>(scale_scratch);
        RCN_CUDA_TRY(cudaMemsetAsync(amax_bits, 0, (size_t)rows * sizeof(unsigned long long), stream));
        // row maxima: of the operand itself, or (im2col columns) of the C channels of the underlying NHWC tensor
        OzOperand am = op;
        int am_rows = rows, am_K = K;
        if (op.gather == 2) {
            am = OzOperand{op.g.t, (size_t)op.g.C, false};
            am_rows = op.g.C;
            am_K = (op.g.n_pix / (op.g.Ho * op.g.Wo)) * op.g.Hi * op.g.Wi;   // every pixel of every image
        }
        int ksplit = (int)((4 * (size_t)kNumSMs + cdiv(am_rows, 32) - 1) / cdiv(am_rows, 32));
        if (ksplit > (am_K + 255) / 256) ksplit = (am_K + 255) / 256;
        if (ksplit < 1) ksplit = 1;
        const int k_per_cta = (am_K + ksplit - 1) / ksplit;
        RCN_LAUNCH("ozaki_amax_rmajor_kernel", stream,
                   ozaki_amax_rmajor_kernel<<<dim3(cdiv(am_rows, 32), (unsigned)ksplit), 256, 0, stream>>>(am, am_rows, am_K, k_per_cta, amax_bits));
        RCN_LAUNCH("ozaki_slice_rmajor_kernel", stream,
                   ozaki_slice_rmajor_kernel<<<dim3(cdiv(rows, 32), cdiv(Kp, RM_KCHUNK)), 256, 0, stream>>>(op, rows, K, Kp, amax_bits,
                                                                                                           planes, scale));
    }
    return RCN_OK;
}

int ozaki_slice_tensor(const double* x, int B, size_t per_image, int8_t* planes, double* scale_out, cudaStream_t stream) {
    if (B <= 0 || per_image == 0) return RCN_OK;
    if (per_image % 64 || (reinterpret_cast<uintptr_t>(x) & 15))
        return fail(RCN_ERR_INVALID, "tensor slicing needs a 16-byte aligned tensor of a multiple of 64 elements per image");
    unsigned long long* amax_bits = reinterpret_cast<unsigned long long*>(scale_out + B);
    RCN_CUDA_TRY(cudaMemsetAsync(amax_bits, 0, (size_t)B * sizeof(unsigned long long), stream));
    // about as many CTAs as the one-scale version launched: up to 8 per SM over the whole tensor
    const unsigned gy = B < 65535 ? (unsigned)B : 65535u;
    unsigned gx = cdiv(per_image, 256 * 8);
    const unsigned gx_max = cdiv((size_t)kNumSMs * 8, gy);
    if (gx > gx_max) gx = gx_max;
    const dim3 grid(gx, gy);
    RCN_LAUNCH("ozaki_amax_tensor_kernel", stream, ozaki_amax_tensor_kernel<<<grid, 256, 0, stream>>>(x, B, per_image, amax_bits));
    RCN_LAUNCH("ozaki_slice_tensor_kernel", stream,
               ozaki_slice_tensor_kernel<<<grid, 256, 0, stream>>>(x, B, per_image, amax_bits, planes, scale_out));
    return RCN_OK;
}

int ozaki_make_conv_tensor_map(CUtensorMap* map, const int8_t* planes, int B, int Hi, int Wi, int C, int tw, int th) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(RCN_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)Wi, (cuuint64_t)Hi, (cuuint64_t)B, (cuuint64_t)OZ_S};
    const cuuint64_t strides[4] = {(cuuint64_t)C, (cuuint64_t)Wi * C, (cuuint64_t)Hi * Wi * C, (cuuint64_t)B * Hi * Wi * C};
    const cuuint32_t box[5] = {(cuuint32_t)OZ_BK, (cuuint32_t)tw, (cuuint32_t)th, 1, 1};
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 5, const_cast<int8_t*>(planes), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS)
        return fail(RCN_ERR_CUDA, "cuTensorMapEncodeTiled (conv) failed with CUresult %d (B %d, H %d, W %d, C %d, box %d x %d)", (int)rc, B, Hi, Wi, C, tw, th);
    return RCN_OK;
}

int ozaki_make_tensor_map(CUtensorMap* map, const int8_t* planes, int rows, int Kp, int box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(RCN_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[3] = {(cuuint64_t)Kp, (cuuint64_t)rows, (cuuint64_t)OZ_S};
    const cuuint64_t strides[2] = {(cuuint64_t)Kp, (cuuint64_t)rows * (cuuint64_t)Kp};   // bytes, dims 1 and 2
    const cuuint32_t box[3] = {(cuuint32_t)OZ_BK, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(planes), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) return fail(RCN_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows %d, Kp %d)", (int)rc, rows, Kp);
    return RCN_OK;
}

}  // namespace rcn
