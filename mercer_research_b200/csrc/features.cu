// features.cu -- rcn's feature stage on sm_100a: separable Sobel x4 -> ReLU -> 2x2 max-pool stacks, flatten,
// standardise.  Reference: rcn/src/utils/kernel.rs:38-53,110-349 and rcn/src/rcn.rs:41-46,230-251,317-356,
// 407-412.  HBM-bound integer/byte work: one image per CTA iteration, all intermediate maps stay in shared
// memory, the only global traffic is the image read and the feature write (SURVEY.md 8d: H*W*s_in + L*8 B).
#include "features.cuh"

#include <type_traits>

#include <cmath>
#include <cstdlib>

namespace rcn {

// ------------------------------------------------------------------------------------------------
// Plan
// ------------------------------------------------------------------------------------------------
int plan_features(const int32_t* cfg, size_t n_cfg, size_t H, size_t W, FeaturePlan* plan) {
    FeaturePlan p;
    p.stages.n = 0;
    size_t maps = 0, h = H, w = W;
    p.max_elems = H * W;
    for (size_t i = 0; i < n_cfg; ++i) {
        const int layer = cfg[i];
        if (layer == RCN_LAYER_CONV_NONE || layer == RCN_LAYER_CONV_SAME) {
            if (h < 3 || w < 3)  // kernel.rs:199-201
                return fail(RCN_ERR_SHAPE,
                            "convolve_2d_separated expects 'self.shape() >= kernel_shape() > 0', received (%zu, %zu) and (3, 3) respectively.", h, w);
            if (p.stages.n >= kMaxStages) return fail(RCN_ERR_INVALID, "convpool stack too deep (max %d stages)", kMaxStages);
            Stage& s = p.stages.s[p.stages.n++];
            s.kind = 0;
            s.same = (layer == RCN_LAYER_CONV_SAME);
            s.first = (maps == 0);
            s.n_in = maps ? (int)maps : 1;
            s.h_in = (int)h; s.w_in = (int)w;
            if (!s.same) { h -= 2; w -= 2; }
            s.h_c = (int)h; s.w_c = (int)w;
            s.h_out = s.h_c; s.w_out = s.w_c;
            maps = maps ? maps * 4 : 4;
            s.n_out = (int)maps;
            p.n_conv++;
            // fuse a directly following pool layer
            if (i + 1 < n_cfg && (cfg[i + 1] == RCN_LAYER_POOL_MAX || cfg[i + 1] == RCN_LAYER_POOL_AVERAGE)) {
                if (cfg[i + 1] == RCN_LAYER_POOL_AVERAGE) return fail(RCN_ERR_NOT_IMPLEMENTED, "Not implemented");  // kernel.rs:284
                if (h < 2 || w < 2)  // kernel.rs:246-251
                    return fail(RCN_ERR_SHAPE, "stride_2d expected a matrix with dimensions greater than (2, 2), got (%zu, %zu)", h, w);
                h = (h + 1) / 2; w = (w + 1) / 2;  // always Padding::Same (rcn.rs:344)
                s.kind = 1;
                s.h_out = (int)h; s.w_out = (int)w;
                ++i;
            }
        } else if (layer == RCN_LAYER_POOL_MAX || layer == RCN_LAYER_POOL_AVERAGE) {
            if (maps == 0) continue;  // pooling an empty feature set is a no-op (rcn.rs:343)
            if (h < 2 || w < 2)
                return fail(RCN_ERR_SHAPE, "stride_2d expected a matrix with dimensions greater than (2, 2), got (%zu, %zu)", h, w);
            if (layer == RCN_LAYER_POOL_AVERAGE) return fail(RCN_ERR_NOT_IMPLEMENTED, "Not implemented");
            if (p.stages.n >= kMaxStages) return fail(RCN_ERR_INVALID, "convpool stack too deep (max %d stages)", kMaxStages);
            Stage& s = p.stages.s[p.stages.n++];
            s.kind = 2; s.same = 1; s.first = 0;
            s.n_in = (int)maps; s.h_in = (int)h; s.w_in = (int)w; s.h_c = (int)h; s.w_c = (int)w;
            h = (h + 1) / 2; w = (w + 1) / 2;
            s.h_out = (int)h; s.w_out = (int)w; s.n_out = (int)maps;
        } else {
            return fail(RCN_ERR_INVALID, "unknown RCNLayer code %d", layer);
        }
        const size_t in_elems = (size_t)p.stages.s[p.stages.n - 1].n_in * p.stages.s[p.stages.n - 1].h_in * p.stages.s[p.stages.n - 1].w_in;
        if (in_elems > p.max_elems) p.max_elems = in_elems;
        if (maps * h * w > ((size_t)1 << 30)) return fail(RCN_ERR_INVALID, "feature set too large");
    }
    p.n_maps = maps; p.map_h = maps ? h : 0; p.map_w = maps ? w : 0;
    p.L = maps * p.map_h * p.map_w;
    *plan = p;
    return RCN_OK;
}

}  // namespace rcn

#include "features_device.cuh"

namespace rcn {

// ------------------------------------------------------------------------------------------------
// Fused path: whole convpool stack of one image in shared memory.
// ------------------------------------------------------------------------------------------------
template <typename TIN, typename T>
__global__ void __launch_bounds__(256) features_fused_kernel(const TIN* __restrict__ images, int B, int H, int W,
                                                            const __grid_constant__ StageList sl, int buf_elems,
                                                            double* __restrict__ out, size_t L, const Standardise sc,
                                                            const BatchIndex bi) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* buf0 = reinterpret_cast<T*>(smem_raw);
    T* buf1 = buf0 + buf_elems;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int img = blockIdx.x; img < B; img += gridDim.x) {
        const size_t src = source_image(bi, (size_t)img);
        if (tid == 0 && bi.labels_batch) bi.labels_batch[img] = bi.labels_all[src];
        load_image<TIN, T>(images + image_slot(bi, src) * H * W, buf0, H, W, tid, nt);
        __syncthreads();
        T* cur = buf0;
        T* nxt = buf1;
        for (int s = 0; s < sl.n; ++s) {
            const Stage& st = sl.s[s];
            if (s == sl.n - 1) {
                EmitFeatures<T> e{out + (size_t)img * L, st.h_out, st.h_out * st.w_out, sc};
                run_stage<T>(st, cur, e, tid, nt);
            } else {
                EmitMaps<T> e{nxt, st.h_out, st.h_out * st.w_out};
                run_stage<T>(st, cur, e, tid, nt);
                __syncthreads();
                T* tmp = cur; cur = nxt; nxt = tmp;
            }
        }
        __syncthreads();  // the next image overwrites buf0
    }
}

// ------------------------------------------------------------------------------------------------
// Staged path for the canonical stacks -- u8 images through [Convolve2D(Same), Pool2D(Max)]^n (main.rs:53-59) --
// built for HBM bandwidth: a persistent CTA pulls its next image into shared memory with one bulk-async copy
// (cp.async.bulk + mbarrier, double-buffered) while it works on the current one; every map lives in shared memory as
// an int32 column-major tile with a zero frame (2 rows above / left, >= 1 below / right, and the never-read last
// column of SURVEY.md A.2 kept at zero), so the 4x4 patch of a pooled output is eight aligned, conflict-free 8-byte
// loads without a single bounds test; the only global traffic is the image read and the coalesced feature write.
// Arithmetic is the same exact int32 closed form as conv_pool_same_int (bit-identical to the reference's f64).
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) features_cp_kernel(const uint8_t* __restrict__ images, int B, int H, int W,
                                                         const __grid_constant__ CpPlan cp, double* __restrict__ out,
                                                         size_t L, const Standardise sc, const BatchIndex bi, int bulk) {
    extern __shared__ __align__(128) unsigned char cp_smem[];
    __shared__ __align__(8) uint64_t bar[2];
    uint8_t* stg0 = cp_smem;
    uint8_t* stg1 = cp_smem + cp.stage_bytes;
    int* tiles = reinterpret_cast<int*>(cp_smem + 2 * cp.stage_bytes);
    const int tid = threadIdx.x, nt = blockDim.x;
    const uint32_t img_bytes = (uint32_t)(H * W);

    for (int i = tid; i < cp.tile_ints; i += nt) tiles[i] = 0;   // the zero frames are written once per CTA
    if (tid == 0) {
        cpbulk::mbar_init(bar + 0, 1);
        cpbulk::mbar_init(bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    int img = blockIdx.x;
    if (bulk && tid == 0 && img < B) {
        const size_t src = source_image(bi, (size_t)img);
        cpbulk::mbar_expect_tx(bar + 0, img_bytes);
        cpbulk::bulk_load(stg0, images + image_slot(bi, src) * img_bytes, img_bytes, bar + 0);
    }
    for (int k = 0; img < B; img += gridDim.x, ++k) {
        const int s = k & 1;
        uint8_t* stg = s ? stg1 : stg0;
        if (bulk) {
            const int nimg = img + gridDim.x;
            if (tid == 0) {
                if (bi.labels_batch) bi.labels_batch[img] = bi.labels_all[source_image(bi, (size_t)img)];
                if (nimg < B) {   // the other staging buffer was drained before the barriers of iteration k-1
                    const size_t nsrc = source_image(bi, (size_t)nimg);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads -> async-proxy overwrite
                    cpbulk::mbar_expect_tx(bar + (s ^ 1), img_bytes);
                    cpbulk::bulk_load(s ? stg0 : stg1, images + image_slot(bi, nsrc) * img_bytes, img_bytes, bar + (s ^ 1));
                }
            }
            cpbulk::mbar_wait(bar + s, (uint32_t)((k >> 1) & 1));
        } else {   // unaligned source: plain loads into the staging buffer
            const size_t src = source_image(bi, (size_t)img);
            if (tid == 0 && bi.labels_batch) bi.labels_batch[img] = bi.labels_all[src];
            const uint8_t* g = images + image_slot(bi, src) * img_bytes;
            for (int i = tid; i < (int)img_bytes; i += nt) stg[i] = g[i];
            __syncthreads();
        }
        cp_transpose_images(stg, 0, tiles, 0, 1, H, W, cp, tid, nt);
        __syncthreads();
        CpSinkGlobal<MODE> sink{out + (size_t)img * L, sc};
        if (cp.n == 1) {
            for (int it = tid; it < cp.s[0].n_in * cp.s[0].h_out * cp.s[0].w_out; it += nt)
                cp_item<true, true>(cp.s[0], tiles, it, nullptr, 0, 0, sink);
        } else {
            for (int it = tid; it < cp.s[0].h_out * cp.s[0].w_out; it += nt)
                cp_item<false, true>(cp.s[0], tiles, it, tiles + cp.s[1].off, cp.s[1].hp, cp.s[1].map_elems, sink);
            __syncthreads();
            for (int q = 1; q < cp.n - 1; ++q) {
                const CpStage& st = cp.s[q];
                const CpStage& nx = cp.s[q + 1];
                for (int it = tid; it < st.n_in * st.h_out * st.w_out; it += nt)
                    cp_item<false, false>(st, tiles + st.off, it, tiles + nx.off, nx.hp, nx.map_elems, sink);
                __syncthreads();   // the next stage reads what this one wrote
            }
            const CpStage& st = cp.s[cp.n - 1];
            for (int it = tid; it < st.n_in * st.h_out * st.w_out; it += nt)
                cp_item<true, false>(st, tiles + st.off, it, nullptr, 0, 0, sink);
        }
        __syncthreads();   // the next image's transpose reuses tile 0
    }
}

// Host: can this plan take the staged path, and with which geometry?
static unsigned cp_magic(unsigned d) { return (unsigned)(0xFFFFFFFFu / d) + 1u; }   // d >= 2
bool make_cp_plan(const FeaturePlan& plan, size_t H, size_t W, CpPlan* out) {
    const StageList& sl = plan.stages;
    if (sl.n < 1 || sl.n > kCpMaxStages || plan.n_conv > 10 || (W & 3) != 0) return false;
    CpPlan cp{};
    cp.n = sl.n;
    size_t off = 0;
    for (int q = 0; q < sl.n; ++q) {
        const Stage& s = sl.s[q];
        if (s.kind != 1 || !s.same) return false;
        CpStage& c = cp.s[q];
        c.n_in = s.n_in; c.h = s.h_in; c.w = s.w_in;
        c.hp = cp_pitch(s.h_in);
        c.map_elems = c.hp * cp_cols(s.w_in);
        c.h_out = s.h_out; c.w_out = s.w_out;
        c.off = (int)off;
        if (s.h_out < 2) return false;   // cp_div needs divisors >= 2; 1-row maps take the generic kernel
        c.magic_hw = cp_magic((unsigned)(s.h_out * s.w_out));
        c.magic_h = cp_magic((unsigned)s.h_out);
        c.magic_items = cp_magic((unsigned)(c.n_in * s.h_out * s.w_out));
        off += (size_t)c.n_in * c.map_elems;
        if ((size_t)c.n_in * s.h_out * s.w_out >= (1u << 16) || off > (1u << 20)) return false;   // cp_div range
    }
    cp.tile_ints = (int)off;
    cp.stage_bytes = (int)((H * W + 127) / 128 * 128);
    cp.magic_w4 = W / 4 >= 2 ? cp_magic((unsigned)(W / 4)) : 0;
    const unsigned chunks = (unsigned)((W / 4 + kCpWordsPerTask - 1) / kCpWordsPerTask);
    cp.magic_chunks = chunks >= 2 ? cp_magic(chunks) : 0;
    cp.tasks_per_image = (int)(((H + 31) / 32) * chunks);
    cp.magic_tasks = cp.tasks_per_image >= 2 ? cp_magic((unsigned)cp.tasks_per_image) : 0;
    *out = cp;
    return true;
}

// ------------------------------------------------------------------------------------------------
// Layer-by-layer path (map sets too large for shared memory): same stage code over global buffers.
// ------------------------------------------------------------------------------------------------
template <typename TIN, typename T>
__global__ void convert_images_kernel(const TIN* __restrict__ images, T* __restrict__ out, int H, int W, size_t B,
                                      const BatchIndex bi) {
    for (size_t img = blockIdx.y; img < B; img += gridDim.y) {
        const size_t src = source_image(bi, img);
        if (blockIdx.x == 0 && threadIdx.x == 0 && bi.labels_batch) bi.labels_batch[img] = bi.labels_all[src];
        load_image<TIN, T>(images + image_slot(bi, src) * H * W, out + img * H * W, H, W, blockIdx.x * blockDim.x + threadIdx.x,
                           gridDim.x * blockDim.x);
    }
}

template <typename T>
__global__ void __launch_bounds__(256) stage_maps_kernel(const __grid_constant__ Stage st, const T* __restrict__ in,
                                                        size_t in_stride, T* __restrict__ out, size_t out_stride, size_t B) {
    for (size_t img = blockIdx.y; img < B; img += gridDim.y) {
        EmitMaps<T> e{out + img * out_stride, st.h_out, st.h_out * st.w_out};
        run_stage<T>(st, in + img * in_stride, e, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    }
}

template <typename T>
__global__ void __launch_bounds__(256) stage_final_kernel(const __grid_constant__ Stage st, const T* __restrict__ in,
                                                         size_t in_stride, double* __restrict__ out, size_t L,
                                                         const Standardise sc, size_t B) {
    for (size_t img = blockIdx.y; img < B; img += gridDim.y) {
        EmitFeatures<T> e{out + img * L, st.h_out, st.h_out * st.w_out, sc};
        run_stage<T>(st, in + img * in_stride, e, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    }
}

// Convolve2D(Same) WITHOUT a pool, exact int32 maps (the wide conv stacks of BASELINE config 4: 64x64 maps fanned out x4 per
// layer stay too large for shared memory, so the stage streams HBM -> HBM).  One CTA = one input map of one image; a thread
// owns output row y and slides a three-column window along x: the vertical passes [1,0,-1] / [1,2,1] of a column are computed
// once and reused by the three outputs that read it, so a pixel costs 3 coalesced loads (lanes = consecutive rows of the
// column-major map) and ~12 integer operations instead of the 9 bounds-tested loads and two integer divisions of the generic
// item loop.  Same closed form as sobel4<int, true> (SURVEY.md A.2: response centred at (y-1, x-1), row 0 zero, last input
// column never read), so the result is bit-identical.
template <typename Emit>
__device__ __forceinline__ void conv_same_strips(const Stage& st, const int* __restrict__ f, int i, const Emit& emit, int tid) {
    const int h = st.h_in, w = st.w_in;
    const int rows = min(h, 256);
    const int n_strips = max(1, 256 / rows);
    const int sw = (w + n_strips - 1) / n_strips;
    const int yl = tid % rows, sidx = tid / rows;
    if (sidx >= n_strips) return;
    const int xa = sidx * sw, xb = min(w, xa + sw);
    int sT, sL, sR, sB;   // slot order rcn.rs:325-339
    if (st.first) { sT = 0; sL = 1; sR = 2; sB = 3; }
    else { sB = i; sT = st.n_in + 3 * i; sL = sT + 1; sR = sT + 2; }
    for (int y = yl; y < h; y += rows) {
        if (y == 0) {
            for (int x = xa; x < xb; ++x) { emit(sT, 0, x, 0); emit(sL, 0, x, 0); emit(sR, 0, x, 0); emit(sB, 0, x, 0); }
            continue;
        }
        const int rr = y - 1;
        auto column = [&](int j, int& ct, int& cs) {
            if (j >= 0 && j <= w - 2) {
                const int* col = f + (size_t)j * h + rr;
                const int a = (rr >= 1) ? col[-1] : 0, b = col[0], c = col[1];
                ct = a - c;            // [1, 0, -1]
                cs = a + 2 * b + c;    // [1, 2, 1]
            } else {
                ct = 0; cs = 0;
            }
        };
        int ct0, cs0, ct1, cs1;
        column(xa - 2, ct0, cs0);
        column(xa - 1, ct1, cs1);
#pragma unroll 2   // (unroll 4 cost 128 registers = two CTAs per SM: 22 % warps active, slower than the generic loop)
        for (int x = xa; x < xb; ++x) {
            int ct2, cs2;
            column(x, ct2, cs2);
            const int t = ct0 + 2 * ct1 + ct2;   // Top; Bottom is its negation
            const int l = cs0 - cs2;             // Left; Right is its negation
            emit(sT, y, x, max(t, 0));
            emit(sL, y, x, max(l, 0));
            emit(sR, y, x, max(-l, 0));
            emit(sB, y, x, max(-t, 0));
            ct0 = ct1; cs0 = cs1; ct1 = ct2; cs1 = cs2;
        }
    }
}

// The CTA's input map is first copied into shared memory (when it fits: `staged`; 16-byte loads, every request of the map
// in flight at once), so the HBM / L2 latency is paid once per map instead of once per pixel (ncu of the first version:
// 57 % of the samples were long-scoreboard waits on the three loads of a pixel).
__device__ __forceinline__ const int* conv_same_stage_map(const int* __restrict__ g, int n, int staged, int* s_map) {
    if (!staged) return g;
    __syncthreads();   // the previous image's map has been consumed
    const int4* g4 = reinterpret_cast<const int4*>(g);
    int4* s4 = reinterpret_cast<int4*>(s_map);
    for (int k = threadIdx.x; k < n / 4; k += 256) s4[k] = g4[k];
    __syncthreads();
    return s_map;
}

__global__ void __launch_bounds__(256, 4) conv_same_maps_kernel(const __grid_constant__ Stage st, const int* __restrict__ in,
                                                            size_t in_stride, int* __restrict__ out, size_t out_stride, size_t B,
                                                            int staged) {
    extern __shared__ __align__(16) int s_map[];
    const int i = blockIdx.x;
    for (size_t img = blockIdx.y; img < B; img += gridDim.y) {
        EmitMaps<int> e{out + img * out_stride, st.h_out, st.h_out * st.w_out};
        const int* f = conv_same_stage_map(in + img * in_stride + (size_t)i * st.h_in * st.w_in, st.h_in * st.w_in, staged, s_map);
        conv_same_strips(st, f, i, e, threadIdx.x);
    }
}

// 4 CTAs per SM (64 registers).  The 40-register build (6 CTAs per SM) measured slower (351 vs 311 us for the c4 stack): more
// resident warps do not help a kernel whose stores already cover DRAM's write rate, and the tighter register budget costs
// instructions.
__global__ void __launch_bounds__(256, 4) conv_same_final_kernel(const __grid_constant__ Stage st, const int* __restrict__ in,
                                                      size_t in_stride, double* __restrict__ out, size_t L,
                                                      const Standardise sc, size_t B, int staged) {
    extern __shared__ __align__(16) int s_map[];
    const int i = blockIdx.x;
    for (size_t img = blockIdx.y; img < B; img += gridDim.y) {
        EmitFeatures<int> e{out + img * L, st.h_out, st.h_out * st.w_out, sc};
        const int* f = conv_same_stage_map(in + img * in_stride + (size_t)i * st.h_in * st.w_in, st.h_in * st.w_in, staged, s_map);
        conv_same_strips(st, f, i, e, threadIdx.x);
    }
}

constexpr size_t kFusedSmemLimit = 200 * 1024;

// u8 images through conv(Same)+pool stacks: the staged kernel above.  Returns false when the plan does not qualify.
static bool try_launch_features_cp(const FeaturePlan& plan, const uint8_t* images, size_t B, size_t H, size_t W,
                                   const Standardise& sc, double* out, cudaStream_t stream, const BatchIndex& bi, int* rc) {
    static const bool off = []() { const char* e = getenv("RCN_CUDA_FEATURES_STAGED"); return e && e[0] == '0'; }();
    CpPlan cp;
    if (off || !make_cp_plan(plan, H, W, &cp)) return false;
    const size_t smem = 2 * (size_t)cp.stage_bytes + (size_t)cp.tile_ints * sizeof(int);
    if (smem > kFusedSmemLimit) return false;
    auto launch = [&]() -> int {
        auto kern = sc.mode == 0 ? features_cp_kernel<0> : sc.mode == 1 ? features_cp_kernel<1> : features_cp_kernel<2>;
        static SmemAttrCache attr[3];
        if (smem > 48 * 1024 && attr[sc.mode].need(smem))
            RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        size_t per_sm = (220 * 1024) / (smem + 1024);
        if (per_sm > 8) per_sm = 8;
        if (per_sm < 1) per_sm = 1;
        size_t grid = (size_t)kNumSMs * per_sm;
        if (grid > B) grid = B;
        const int bulk = ((H * W) % 16 == 0 && (reinterpret_cast<uintptr_t>(images) % 16) == 0) ? 1 : 0;
        RCN_LAUNCH("features_cp_kernel", stream,
                   kern<<<(unsigned)grid, 256, smem, stream>>>(images, (int)B, (int)H, (int)W, cp, out, plan.L, sc, bi, bulk));
        return RCN_OK;
    };
    *rc = launch();
    return true;
}

template <typename TIN, typename T>
static int launch_features_t(const FeaturePlan& plan, const TIN* images, size_t B, size_t H, size_t W,
                             const Standardise& sc, double* out, FeatureScratch& scratch, cudaStream_t stream,
                             const BatchIndex& bi) {
    const StageList& sl = plan.stages;
    const size_t smem = 2 * plan.max_elems * sizeof(T);
    if (smem <= kFusedSmemLimit) {
        auto kern = features_fused_kernel<TIN, T>;
        if (smem > 48 * 1024) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // One image per CTA iteration; enough CTAs per SM to hide the load -> compute -> store chain.
        size_t per_sm = smem ? (kFusedSmemLimit / smem) : 8;
        if (per_sm > 8) per_sm = 8;
        if (per_sm < 1) per_sm = 1;
        size_t grid = (size_t)kNumSMs * per_sm;
        if (grid > B) grid = B;
        RCN_LAUNCH("features_fused_kernel", stream, kern<<<(unsigned)grid, 256, smem, stream>>>(images, (int)B, (int)H, (int)W, sl, (int)plan.max_elems, out, plan.L,
                                                    sc, bi));
        return RCN_OK;
    }
    // layer-by-layer over global ping-pong buffers
    size_t max_set = H * W;
    for (int s = 0; s < sl.n; ++s) {
        size_t o = (size_t)sl.s[s].n_out * sl.s[s].h_out * sl.s[s].w_out;
        if (s + 1 < sl.n && o > max_set) max_set = o;
    }
    RCN_TRY(scratch.a.reserve(B * max_set * sizeof(T)));
    RCN_TRY(scratch.b.reserve(B * max_set * sizeof(T)));
    T* cur = scratch.a.as<T>();
    T* nxt = scratch.b.as<T>();
    size_t cur_stride = H * W;
    {
        dim3 grid(cdiv(H * W, 256), (unsigned)(B > 32768 ? 32768 : B));
        if (grid.x > 64) grid.x = 64;
        RCN_LAUNCH("convert_images_kernel", stream, convert_images_kernel<TIN, T><<<grid, 256, 0, stream>>>(images, cur, (int)H, (int)W, B, bi));
    }
    for (int s = 0; s < sl.n; ++s) {
        const Stage& st = sl.s[s];
        const size_t items = (size_t)st.n_in * st.h_out * st.w_out;
        dim3 grid(cdiv(items, 256), (unsigned)(B > 32768 ? 32768 : B));
        if (grid.x > 1024) grid.x = 1024;
        if (std::is_same<T, int>::value && st.kind == 0 && st.same && st.h_in >= 2) {   // streaming strip kernels (see above)
            const dim3 sgrid((unsigned)st.n_in, grid.y);
            const int* cin = reinterpret_cast<const int*>(cur);
            // the map goes through shared memory when it fits the default 48 KB and 16-byte loads are possible
            const size_t map_elems = (size_t)st.h_in * st.w_in;
            const int staged = (map_elems * sizeof(int) <= 48 * 1024 && map_elems % 4 == 0 && cur_stride % 4 == 0 &&
                                (reinterpret_cast<uintptr_t>(cin) & 15) == 0) ? 1 : 0;
            const size_t ssmem = staged ? map_elems * sizeof(int) : 0;
            if (s == sl.n - 1) {
                RCN_LAUNCH("conv_same_final_kernel", stream, conv_same_final_kernel<<<sgrid, 256, ssmem, stream>>>(st, cin, cur_stride, out, plan.L, sc, B, staged));
            } else {
                const size_t out_stride = (size_t)st.n_out * st.h_out * st.w_out;
                RCN_LAUNCH("conv_same_maps_kernel", stream, conv_same_maps_kernel<<<sgrid, 256, ssmem, stream>>>(st, cin, cur_stride, reinterpret_cast<int*>(nxt), out_stride, B, staged));
                T* tmp = cur; cur = nxt; nxt = tmp;
                cur_stride = out_stride;
            }
            continue;
        }
        if (s == sl.n - 1) {
            RCN_LAUNCH("stage_final_kernel", stream, stage_final_kernel<T><<<grid, 256, 0, stream>>>(st, cur, cur_stride, out, plan.L, sc, B));
        } else {
            const size_t out_stride = (size_t)st.n_out * st.h_out * st.w_out;
            RCN_LAUNCH("stage_maps_kernel", stream, stage_maps_kernel<T><<<grid, 256, 0, stream>>>(st, cur, cur_stride, nxt, out_stride, B));
            T* tmp = cur; cur = nxt; nxt = tmp;
            cur_stride = out_stride;
        }
    }
    return RCN_OK;
}

// Host check that the 3-instruction Markstein division equals IEEE division for every integer feature value
// 0..vmax with this (mean, sd): makes the fast epilogue provably bit-exact for the u8 pipeline.
static bool standardise_fast_ok(double mean, double sd, long long vmax, double* rcp_out) {
    if (!(sd > 0.0) || !std::isfinite(sd) || !std::isfinite(mean) || vmax > (1ll << 22)) return false;
    const volatile double rcp_v = 1.0 / sd;
    const double rcp = rcp_v;
    for (long long v = 0; v <= vmax; ++v) {
        const double a = (double)v - mean;
        const volatile double exact = a / sd;
        const volatile double q = a * rcp;
        const double rem = std::fma(-q, sd, a);
        const double fast = std::fma(rem, rcp, (double)q);
        const double ex = exact;
        if (std::memcmp(&fast, &ex, sizeof(double)) != 0) return false;
    }
    *rcp_out = rcp;
    return true;
}

Standardise make_standardise(const FeaturePlan& plan, int pixel_format, bool standardise, double mean, double sd) {
    Standardise sc{standardise ? 1 : 0, mean, sd, 0.0};
    if (standardise && pixel_format == RCN_PIXELS_U8_ROWMAJOR && plan.n_conv <= 10) {
        // cache of the last verified (mean, sd, vmax): set_scale is rare, steps are not
        static thread_local double c_mean = 0, c_sd = 0, c_rcp = 0;
        static thread_local long long c_vmax = -1;
        static thread_local bool c_ok = false;
        const long long vmax = 255ll << (2 * plan.n_conv);
        if (!(c_vmax == vmax && c_mean == mean && c_sd == sd)) {
            c_ok = standardise_fast_ok(mean, sd, vmax, &c_rcp);
            c_mean = mean; c_sd = sd; c_vmax = vmax;
        }
        if (c_ok) { sc.mode = 2; sc.rcp = c_rcp; }
    }
    return sc;
}

int launch_features(const FeaturePlan& plan, const void* images, int pixel_format, size_t B, size_t H, size_t W,
                    bool standardise, double mean, double sd, double* out, FeatureScratch& scratch,
                    cudaStream_t stream, const BatchIndex* index) {
    const BatchIndex bi = index ? *index : BatchIndex{};
    if (B == 0 || plan.L == 0) return RCN_OK;  // no conv layer => empty feature vector (rcn.rs:323,339)
    if (B > ((size_t)1 << 30)) return fail(RCN_ERR_INVALID, "batch too large");
    const Standardise sc = make_standardise(plan, pixel_format, standardise, mean, sd);
    if (pixel_format == RCN_PIXELS_U8_ROWMAJOR) {
        // u8 pixels: every intermediate is an integer bounded by 255 * 4^n_conv, so int32 arithmetic is exact
        // (and bit-identical to the reference's f64) up to 10 conv layers.
        int rc = RCN_OK;
        if (try_launch_features_cp(plan, (const uint8_t*)images, B, H, W, sc, out, stream, bi, &rc)) return rc;
        if (plan.n_conv <= 10)
            return launch_features_t<uint8_t, int>(plan, (const uint8_t*)images, B, H, W, sc, out, scratch, stream, bi);
        return launch_features_t<uint8_t, double>(plan, (const uint8_t*)images, B, H, W, sc, out, scratch, stream, bi);
    }
    if (pixel_format == RCN_PIXELS_F64_COLMAJOR)
        return launch_features_t<double, double>(plan, (const double*)images, B, H, W, sc, out, scratch, stream, bi);
    return fail(RCN_ERR_INVALID, "unknown pixel format %d", pixel_format);
}

// ------------------------------------------------------------------------------------------------
// standardise (rcn.rs:407-412) and gen_scales (rcn.rs:230-251)
// ------------------------------------------------------------------------------------------------
__global__ void standardise_kernel(double* __restrict__ v, size_t n, double mean, double sd) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double d = (v[i] - mean) / sd;
        v[i] = (d >= 0.0) ? d : 0.0;
    }
}

int launch_standardise(double* feats, size_t n, double mean, double sd, cudaStream_t stream) {
    if (n == 0) return RCN_OK;
    unsigned grid = cdiv(n, 256);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    RCN_LAUNCH("standardise_kernel", stream, standardise_kernel<<<grid, 256, 0, stream>>>(feats, n, mean, sd));
    return RCN_OK;
}

__device__ __forceinline__ double block_sum_256(double v, double* sm) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double s = 0.0;
    if (warp == 0) {
        s = (lane < (blockDim.x >> 5)) ? sm[lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    }
    __syncthreads();
    return s;  // valid in warp 0
}

// pass == 0: partial sums of v; pass == 1: partial sums of (v - mean)^2 with mean = result[0]
__global__ void __launch_bounds__(256) scale_partial_kernel(const double* __restrict__ v, size_t n, int pass,
                                                           const double* __restrict__ result, double* __restrict__ partial) {
    __shared__ double sm[8];
    const double mean = pass ? result[0] : 0.0;
    double acc = 0.0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double d = v[i] - mean;
        acc += pass ? d * d : d;
    }
    const double s = block_sum_256(acc, sm);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(256) scale_final_kernel(const double* __restrict__ partial, int n_part, size_t n, int pass,
                                                         double* __restrict__ result) {
    __shared__ double sm[8];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n_part; i += blockDim.x) acc += partial[i];
    const double s = block_sum_256(acc, sm);
    if (threadIdx.x == 0) {
        if (pass == 0) result[0] = s / (double)n;          // mean /= n          (rcn.rs:240)
        else result[1] = sqrt(s / (double)n);              // sqrt(sd / n)       (rcn.rs:247)
    }
}

int launch_gen_scales(const double* feats, size_t n, double* result_dev, DevBuf& scratch, cudaStream_t stream) {
    if (n == 0) return fail(RCN_ERR_INVALID, "gen_scales on an empty set");
    int grid = (int)cdiv(n, 256 * 8);
    if (grid > kNumSMs * 4) grid = kNumSMs * 4;
    if (grid < 1) grid = 1;
    RCN_TRY(scratch.reserve((size_t)grid * sizeof(double)));
    double* partial = scratch.as<double>();
    for (int pass = 0; pass < 2; ++pass) {
        RCN_LAUNCH("scale_partial_kernel", stream, scale_partial_kernel<<<grid, 256, 0, stream>>>(feats, n, pass, result_dev, partial));
        RCN_LAUNCH("scale_final_kernel", stream, scale_final_kernel<<<1, 256, 0, stream>>>(partial, grid, n, pass, result_dev));
    }
    return RCN_OK;
}

// ------------------------------------------------------------------------------------------------
// op-level kernels: Convolve2D / Pool2D traits on a single matrix (kernel.rs:61-100, 219-236)
// ------------------------------------------------------------------------------------------------
// convolve_2d (kernel.rs:110-194) with an arbitrary kernel.  Products are not exact here, so multiply and add
// are rounded separately (__dmul_rn / __dadd_rn are never contracted), ky outer / kx inner from +0.
__global__ void conv2d_generic_kernel(const double* __restrict__ m, int H, int W, const double* __restrict__ k, int kh,
                                      int kw, int same, double* __restrict__ out, int oh, int ow) {
    const int ph = same ? kh / 2 : 0, pw = same ? kw / 2 : 0;
    const size_t total = (size_t)oh * ow;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int cx = (int)(idx / oh), cy = (int)(idx - (size_t)cx * oh);
        double acc = 0.0;
        for (int ky = 0; ky < kh; ++ky)
            for (int kx = 0; kx < kw; ++kx) {
                double p;
                if (same) {
                    // padded copy matrix[(cy,cx)] = self[(cy-1,cx-1)] for cy in 1..H+ph, cx in 1..W+pw (kernel.rs:154-158)
                    const int py = cy + ky, px = cx + kx;
                    p = (py >= 1 && py < H + ph && px >= 1 && px < W + pw) ? m[(size_t)(px - 1) * H + (py - 1)] : 0.0;
                } else {
                    p = m[(size_t)(cx + kx) * H + (cy + ky)];
                }
                acc = __dadd_rn(acc, __dmul_rn(p, k[(size_t)kx * kh + ky]));
            }
        out[idx] = acc;
    }
}

int launch_convolve_2d(const double* m, size_t H, size_t W, const double* k, size_t kh, size_t kw, int padding,
                       double* out, cudaStream_t stream) {
    const bool same = padding == RCN_PADDING_SAME;
    const size_t oh = same ? H : H - kh + 1, ow = same ? W : W - kw + 1;
    unsigned grid = cdiv(oh * ow, 256);
    if (grid > kNumSMs * 16) grid = kNumSMs * 16;
    RCN_LAUNCH("conv2d_generic_kernel", stream, conv2d_generic_kernel<<<grid, 256, 0, stream>>>(m, (int)H, (int)W, k, (int)kh, (int)kw, same ? 1 : 0, out, (int)oh, (int)ow));
    return RCN_OK;
}

template <bool SAME>
__global__ void conv_sep_single_kernel(const double* __restrict__ m, int H, int W, int op, double* __restrict__ out, int oh, int ow) {
    const size_t total = (size_t)oh * ow;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx / oh), y = (int)(idx - (size_t)x * oh);
        double t, l, r, b;
        sobel4<double, SAME>(m, H, W, y, x, t, l, r, b);
        const double v = op == RCN_OP_TOP ? t : op == RCN_OP_BOTTOM ? b : op == RCN_OP_LEFT ? l : r;
        out[idx] = relu1(v);
    }
}

int launch_convolve_2d_separated(const double* m, size_t H, size_t W, int op, int padding, double* out, cudaStream_t stream) {
    const bool same = padding == RCN_PADDING_SAME;
    const size_t oh = same ? H : H - 2, ow = same ? W : W - 2;
    unsigned grid = cdiv(oh * ow, 256);
    if (grid > kNumSMs * 16) grid = kNumSMs * 16;
    if (same) RCN_LAUNCH("conv_sep_single_kernel", stream, conv_sep_single_kernel<true><<<grid, 256, 0, stream>>>(m, (int)H, (int)W, op, out, (int)oh, (int)ow));
    else RCN_LAUNCH("conv_sep_single_kernel", stream, conv_sep_single_kernel<false><<<grid, 256, 0, stream>>>(m, (int)H, (int)W, op, out, (int)oh, (int)ow));
    return RCN_OK;
}

__global__ void relu_kernel(const double* __restrict__ m, size_t n, double* __restrict__ out) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = relu1(m[i]);
}

int launch_relu(const double* m, size_t n, double* out, cudaStream_t stream) {
    if (n == 0) return RCN_OK;
    unsigned grid = cdiv(n, 256);
    if (grid > kNumSMs * 16) grid = kNumSMs * 16;
    RCN_LAUNCH("relu_kernel", stream, relu_kernel<<<grid, 256, 0, stream>>>(m, n, out));
    return RCN_OK;
}

// pool_2d (kernel.rs:245-349), Max only.  pad_h/pad_w: zero row/col appended (Padding::Same on odd sizes).
__global__ void pool2d_kernel(const double* __restrict__ m, int H, int W, double* __restrict__ out, int oh, int ow,
                              uint8_t* __restrict__ argmax, int* __restrict__ nan_flag) {
    const size_t total = (size_t)oh * ow;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int rx = (int)(idx / oh), ry = (int)(idx - (size_t)rx * oh);
        double best = 0.0;
        int bi = 0;
        bool nan = false;
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // pooler[py + 2*px] = m[(2ry+px, 2rx+py)]  (kernel.rs:273-277)
            const int cy = 2 * ry + (q >> 1), cx = 2 * rx + (q & 1);
            const double v = (cy < H && cx < W) ? m[(size_t)cx * H + cy] : 0.0;
            nan |= (v != v);
            if (q == 0) { best = v; bi = 0; }
            else if (!(v < best)) { best = v; bi = q; }
        }
        out[idx] = best;
        if (argmax) argmax[idx] = (uint8_t)bi;
        if (nan && nan_flag) *nan_flag = 1;
    }
}

int launch_pool_2d(const double* m, size_t H, size_t W, int padding, double* out, uint8_t* argmax, int* nan_flag,
                   cudaStream_t stream) {
    const bool same = padding == RCN_PADDING_SAME;
    const size_t oh = same ? (H + 1) / 2 : H / 2, ow = same ? (W + 1) / 2 : W / 2;
    if (oh * ow == 0) return RCN_OK;
    unsigned grid = cdiv(oh * ow, 256);
    if (grid > kNumSMs * 16) grid = kNumSMs * 16;
    RCN_LAUNCH("pool2d_kernel", stream, pool2d_kernel<<<grid, 256, 0, stream>>>(m, (int)H, (int)W, out, (int)oh, (int)ow, argmax, nan_flag));
    return RCN_OK;
}

}  // namespace rcn
