// smallnet.cu -- fused training step for rcn's canonical network family: one wide input layer (n_in = feature
// length, e.g. 784) into narrow sigmoid layers (every layer width <= 32, e.g. 784-30-10, main.rs:51-62).
//
// Reference: rcn/src/rcn.rs:317-356 + 407-412 (features), :260-314 (backprop), :176-223 (batch sum), :105-116
// (forward), :152-157 (accuracy).  At these sizes the generic tiled GEMMs of dense.cu are launch/latency bound
// (M = 30 or 10), so a whole minibatch runs as TWO kernels (plus the SGD update):
//
//   A  smallnet_fwd_bwd_kernel   one 16-warp CTA per 8 samples.
//        (fused front end, u8 images) two warps per image run the convpool stack in shared memory with exact
//        int32 arithmetic and write the standardised feature vector both to HBM (kernel B reads it) and into a
//        padded shared-memory tile;
//        z1 = W1 a0 on the f64 tensor path (DMMA.8x8x4): each warp owns a K-range of the 784-deep contraction,
//        streams its W1 fragments straight from L2 into registers and reads the a0 fragments from the tile;
//        partial sums meet in shared memory; the narrow layers (weights prefetched to shared memory), the output
//        delta, the backward-data chain and the batch statistics finish on chip.  Writes a_l, delta_l.
//   B  smallnet_wgrad_kernel     dW1 = Delta1 A0^T over (64-column group) x (K-split of the batch): the Delta1 slice
//        is staged once in shared memory, the A0 fragments stream from L2 with 16 loads in flight per lane, DMMA
//        again; one extra CTA per K-split does db1 and the narrow layers' dW/db.  The last CTA of each column
//        group to finish (atomic ticket) sums the K-split partials in a FIXED order into the flat gradient buffer
//        (the all-reduce target) -- deterministic, unlike the reference's mutex-ordered sum (rcn.rs:190-205).
//
// Data-parallel groups (dp.cu): kernel B pushes its finished sums to the peers, a small exchange kernel X receives, adds and
// updates.  Kernel A of the NEXT step is launched as X's programmatic dependent and runs its whole parameter-independent
// front end (image loads, transpose, conv+pool, feature stores) BEFORE griddepcontrol.wait, i.e. while X is still waiting
// for the NVLink traffic: the exchange leaves the step's critical path.  That is safe because (i) X triggers its
// dependents only after its own wait, so kernel B of the previous step -- the last reader of the feature buffer and the
// writer of the epoch cursor -- has completed and flushed before kernel A's first instruction; (ii) X touches only
// parameters, gradients and its communication block; (iii) X runs as <= 20 fat CTAs, so kernel A's 128 CTAs find an SM each.
#include "smallnet.cuh"
#include "dp.cuh"

#include "features_device.cuh"
#include "timeline.cuh"

#include <cooperative_groups.h>

#include <cstdlib>

namespace rcn {

__device__ __forceinline__ double sn_sigmoid(double z) { return 1.0 / (1.0 + exp(-z)); }  // rcn.rs:478-483

__device__ __forceinline__ void sn_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// Optional phase clock (profiles/sn_phases.py builds a second library with -DRCN_SN_PHASES): thread 0 of every CTA of
// kernel A stamps clock64() at the phase boundaries.  Compiled out of the product library.
#ifdef RCN_SN_PHASES
__device__ long long g_sn_phase[1024][32];
__device__ long long g_snp_stamp[1024][8];
#define SN_PHASE(k) do { if (threadIdx.x == 0 && blockIdx.x < 1024) g_sn_phase[blockIdx.x][k] = clock64(); } while (0)
#else
#define SN_PHASE(k) do { } while (0)
#endif

// Parameter loads.  The default is the read-only path (ld.global.nc).  A PREWAIT kernel is ALIVE while the previous step's
// exchange kernel still rewrites the parameters, which breaks the contract of ld.global.nc ("not modified during the
// kernel's lifetime") -- and ptxas does hoist such loads above griddepcontrol.wait (seen in SASS, round 2: two
// LDG.E.64.CONSTANT of W0 sat in front of ACQBULK and read stale weights; caught by bench.py's graph-replayed parity block).
// There the parameters are read with VOLATILE loads the compiler may not move across the wait: ld.global.cg (L2) for what is
// consumed at once, ld.global.ca for the part of W0 that was prefetched into L1 AFTER the wait (this SM's L1 was
// invalidated when the CTA started and no parameter line entered it before the wait, so it cannot hold a stale one).
// MODE 0: read-only path; 1: volatile .cg; 2: volatile .ca.
template <int MODE>
__device__ __forceinline__ double sn_ld(const double* p) {
    if (MODE == 0) return __ldg(p);
    double v;
    if (MODE == 1) asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    else asm volatile("ld.global.ca.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

constexpr int SN_TB = 8;          // samples per CTA in kernel A (one DMMA n-fragment)
constexpr int SNA_THREADS = 512;  // kernel A
constexpr int SNA_WARPS = 16;
constexpr int SNB_THREADS = 256;  // kernel B
constexpr int SN_TILE_PAD = 4;    // a0 tile row pitch = n_in + 4 doubles: conflict-free B-fragment reads
constexpr int SN_DPITCH = 36;     // delta slice row pitch (doubles): conflict-free A-fragment reads
constexpr int SN_U = 7;           // k-steps of W0 fragments a warp keeps in registers
constexpr int SN_ZPITCH = 36;     // layer-0 partial sums [warp][sample][36]: conflict-free for the DMMA C fragments and the row reads
constexpr int SN_MAX_SMALL = 32 + (kSmallNetMaxLayers - 1) * (32 * 32 + 32);  // params after W0

// final-stage emit of the fused front end: standardised feature -> shared tile + HBM (TO_HBM = false: the tile only)
template <bool TO_HBM>
struct EmitTile {
    double* tile; double* gout; int h, hw; Standardise sc;
    __device__ __forceinline__ void operator()(int slot, int y, int x, int v) const {
        double d = (double)v;
        if (sc.mode == 1) {
            d = (d - sc.mean) / sc.sd;
            d = (d >= 0.0) ? d : 0.0;
        } else if (sc.mode == 2) {  // host-verified exact Markstein division, see EmitFeatures
            const double a = d - sc.mean;
            const double q = __dmul_rn(a, sc.rcp);
            const double rem = fma(-q, sc.sd, a);
            d = fma(rem, sc.rcp, q);
            d = (d >= 0.0) ? d : 0.0;
        }
        const int idx = slot * hw + x * h + y;
        tile[idx] = d;
        if (TO_HBM) gout[idx] = d;
    }
};

// staged front end: standardised feature -> shared tile + HBM
// MAY_DEFER (the PREWAIT kernels): gout == nullptr = only the tile is written here and the HBM copy goes out from the tile once
// griddepcontrol.wait has passed (prewait 2: until then the previous step's kernel B may still be reading the feature buffer).
// Behind the exchange kernel (prewait 1) kernel B has long finished and the copy is written here, off the critical path --
// deferring it there as well cost 2.4 us per step on two GPUs (24.5 vs 22.1).
template <bool MAY_DEFER>
struct CpSinkTile {
    double* tile; double* gout; Standardise sc;
    __device__ __forceinline__ void operator()(int idx, int v) const {
        const double d = cp_finish(sc.mode, v, sc);
        tile[idx] = d;
        if (!MAY_DEFER || gout) gout[idx] = d;
    }
};

__device__ __forceinline__ unsigned char* sn_align128(void* p) {
    return reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(p) + 127) & ~(uintptr_t)127);
}

// What the inference variant of kernel A (smallnet_infer_kernel) writes besides its per-tile {cost, hits} partials.
struct SnInfer {
    int64_t* labels_out;     // optional: argmax of every sample (argmax_last_kernel's rule)
    unsigned* ticket;        // zero before the launch; the last CTA resets it
    double* stats;           // {cost, hits as uint64 bits} of the launch
    int accumulate;          // add to stats instead of overwriting them (the chunks of a batch above smallnet_max_batch())
};

// ------------------------------------------------------------------------------------------------
// Kernel A
// ------------------------------------------------------------------------------------------------
// FUSED 0: features are an input; 1: generic fused front end; 2: staged front end (CpPlan).
// PREWAIT (FUSED == 2, data-parallel groups): the whole front end runs before griddepcontrol.wait -- under the previous
// step's exchange kernel -- and only the parameter loads wait for it (see the file header for why that is safe).
// INFER (smallnet_infer_kernel, backward == 0): forward only, nothing but the statistics partials, `inf.stats` and
// `inf.labels_out` goes to global memory -- the features stay in the shared tile and the activations on chip.
template <int FUSED, bool PREWAIT, bool INFER>
__device__ __forceinline__ void sn_phase_a(const SmallNetDesc& d, const double* __restrict__ params,
                                           double* __restrict__ feats, int B, const double* __restrict__ onehot,
                                           const int64_t* __restrict__ labels, double* __restrict__ acts,
                                           double* __restrict__ deltas, double* __restrict__ stats_partial,
                                           int backward, const SmallNetFront& fr,
                                           const int tile_idx, unsigned char* sn_smem, const SnInfer& inf) {
    double* zpart = reinterpret_cast<double*>(sn_smem);                 // [16][8][36]
    double* s_small = zpart + SNA_WARPS * SN_TB * SN_ZPITCH;                   // params after W0: b0 | W1 | b1 | ...
    double* tile = s_small + SN_MAX_SMALL;                              // FUSED: [8][n_in + 4]
    __shared__ double s_act[kSmallNetMaxLayers][SN_TB][33];
    __shared__ double s_del[kSmallNetMaxLayers][SN_TB][33];
    __shared__ double s_cost[SN_TB];
    __shared__ unsigned long long s_hit[SN_TB];
    __shared__ long long s_label[SN_TB];

    // programmatic dependent launch (when the host asked for it; no-ops otherwise): let the next kernel's launch proceed
    // under this one, and wait until the previous kernel has completed and flushed before touching global memory
    // (a forward-only launch keeps the implicit trigger at its completion: its successor may be a PREWAIT kernel A, whose
    // early part writes the feature buffer)
    if (backward) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (!PREWAIT) asm volatile("griddepcontrol.wait;" ::: "memory");
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int s0 = tile_idx * SN_TB;
    const int L = d.n_in, R0 = d.rows[0];
    const int mf = (R0 + 7) >> 3;
    SN_PHASE(0);
    RCN_TL_BEGIN(d.tl, 0);
    const int pitch = L + SN_TILE_PAD;
    const int small_base = d.b_off[0];
    const int n_small = d.n_params - small_base;

    // staged front end: the image loads go out before anything else asks the memory system for data
    __shared__ __align__(8) uint64_t s_bar;
    unsigned char* stg = sn_align128(tile + SN_TB * pitch);
    if (FUSED == 2) {
        const int n_live = min(SN_TB, B - s0);
        const uint32_t img_bytes = (uint32_t)(fr.H * fr.W);
        if (warp == 0) {
            if (lane == 0) {
                cpbulk::mbar_init(&s_bar, 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
                cpbulk::mbar_expect_tx(&s_bar, img_bytes * (uint32_t)n_live);
            }
            __syncwarp();
            if (lane < n_live) {
                const size_t src = source_image(fr.bi, (size_t)(s0 + lane));
                wait_arrived(fr.bi, src);
                cpbulk::bulk_load(stg + lane * fr.cp.stage_bytes, fr.images + image_slot(fr.bi, src) * img_bytes, img_bytes, &s_bar);
            }
        } else if (warp == SNA_WARPS - 1 && lane < SN_TB) {
            // the labels take a second dependent global load: another warp fetches them, off warp 0's critical path
            long long lab = -1;
            if (lane < n_live) {
                const int sample = s0 + lane;
                const size_t src = source_image(fr.bi, (size_t)sample);
                lab = fr.bi.cursor ? fr.bi.labels_all[src] : (labels ? labels[sample] : 0);
                if (fr.bi.labels_batch) fr.bi.labels_batch[sample] = lab;
            }
            s_label[lane] = lab;
        }
    }

    SN_PHASE(8);
    // layer-0 weight fragments: each warp owns a K range of the n_in-deep contraction; its first SN_U k-steps go into
    // registers NOW and the rest is prefetched into L1, so the L2 latency is hidden behind the front end (PREWAIT: the
    // parameters are not final yet -- the same loads are issued right after the wait below instead)
    const double* __restrict__ W0 = params + d.w_off[0];
    const int ksteps = (L + 3) >> 2;
    const int per_warp = (ksteps + SNA_WARPS - 1) / SNA_WARPS;
    const int ks_begin = warp * per_warp;
    const int ks_end = min(ksteps, ks_begin + per_warp);
    bool rowok[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) rowok[i] = (i < mf) && (i * 8 + g < R0);
    double w_pre[SN_U][4];
    auto load_params = [&]() {
#pragma unroll
        for (int u = 0; u < SN_U; ++u) {
            const int k = (ks_begin + u) * 4 + t;
            const bool kok = (ks_begin + u) < ks_end && k < L;
            const double* wp = W0 + (size_t)k * R0 + g;
#pragma unroll
            for (int i = 0; i < 4; ++i) w_pre[u][i] = (kok && rowok[i]) ? sn_ld<PREWAIT ? 1 : 0>(wp + i * 8) : 0.0;  // A frag: row g (m), col t (k)
        }
        SN_PHASE(9);
        // biases + narrow-layer weights into shared memory (after the register loads above), as asynchronous copies: no
        // register dependency, so no warp waits an L2 round trip here (PREWAIT: through registers, coherent at L2)
        if (PREWAIT) {
            for (int i = tid; i < n_small; i += SNA_THREADS) s_small[i] = sn_ld<1>(params + small_base + i);
        } else {
            for (int i = tid; i < n_small; i += SNA_THREADS) {
                const unsigned dst = (unsigned)__cvta_generic_to_shared(s_small + i);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(params + small_base + i) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        // the rest of this warp's K range of W0 into L1
        const long long lo = (long long)min((ks_begin + SN_U) * 4, L) * R0, hi = (long long)min(ks_end * 4, L) * R0;   // doubles
        for (long long e = lo + lane * 16; e < hi; e += 32 * 16)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(W0 + e) : "memory");
    };
    if (!PREWAIT) load_params();

    if (FUSED == 2) {
        // ---- staged front end: the 8 images arrive by bulk-async copies while the tiles' zero frames are written; then
        // all 16 warps transpose and run the conv+pool stages over the 8 images together (features_device.cuh) ---------
        // (fr.cp_pairs: SN_TB / 2 packed tiles, pair q = images q and q + SN_TB / 2, see cp_item_pair)
        int* tiles = reinterpret_cast<int*>(stg + SN_TB * fr.cp.stage_bytes);
        const int n_live = min(SN_TB, B - s0);
        const int n_tiles = fr.cp_pairs ? SN_TB / 2 : SN_TB;
        SN_PHASE(10);
        for (int i = tid; i < n_tiles * fr.cp.tile_ints; i += SNA_THREADS) tiles[i] = 0;
        for (int i = n_live * pitch + tid; i < SN_TB * pitch; i += SNA_THREADS) tile[i] = 0.0;   // absent samples
        SN_PHASE(11);
        __syncthreads();
        SN_PHASE(12);
        cpbulk::mbar_wait(&s_bar, 0u);
        SN_PHASE(1);
        if (fr.cp_pairs)
            cp_transpose_pairs(stg, fr.cp.stage_bytes, SN_TB / 2, reinterpret_cast<uint32_t*>(tiles), fr.cp.tile_ints, n_live,
                               fr.H, fr.W, fr.cp, tid, SNA_THREADS);
        else
            cp_transpose_images(stg, fr.cp.stage_bytes, tiles, fr.cp.tile_ints, n_live, fr.H, fr.W, fr.cp, tid, SNA_THREADS);
        __syncthreads();
        SN_PHASE(2);
        if (fr.cp_pairs) {
            const CpStage& st = fr.cp.s[0];
            const int items = st.h_out * st.w_out;
            for (int it = tid; it < min(SN_TB / 2, n_live) * items; it += SNA_THREADS) {
                const int q = cp_div(it, st.magic_items);   // one input map: magic_items divides by h_out * w_out
                const int itl = it - q * items;
                const int qy = q + SN_TB / 2;
                const bool live_y = qy < n_live;
                const bool hbm = !(INFER || (PREWAIT && fr.prewait == 2));
                CpSinkTile<PREWAIT || INFER> sx{tile + (size_t)q * pitch, hbm ? feats + (size_t)(s0 + q) * L : nullptr, fr.sc};
                CpSinkTile<PREWAIT || INFER> sy{tile + (size_t)qy * pitch, hbm && live_y ? feats + (size_t)(s0 + qy) * L : nullptr,
                                                fr.sc};
                cp_item_pair(st, reinterpret_cast<const uint32_t*>(tiles) + q * fr.cp.tile_ints, itl, sx, sy, live_y);
            }
            __syncthreads();
        } else {
            for (int q = 0; q < fr.cp.n; ++q) {
                const CpStage& st = fr.cp.s[q];
                const int items = st.n_in * st.h_out * st.w_out;
                const bool last = q == fr.cp.n - 1;
                const CpStage& nx = fr.cp.s[last ? q : q + 1];
                for (int it = tid; it < n_live * items; it += SNA_THREADS) {
                    const int gi = cp_div(it, st.magic_items);
                    const int itl = it - gi * items;
                    const int* in = tiles + gi * fr.cp.tile_ints + st.off;
                    int* nxt = tiles + gi * fr.cp.tile_ints + nx.off;
                    CpSinkTile<PREWAIT || INFER> sink{tile + (size_t)gi * pitch,
                                                      (INFER || (PREWAIT && fr.prewait == 2)) ? nullptr : feats + (size_t)(s0 + gi) * L, fr.sc};
                    if (last) {   // q > 0: one-stage plans take the packed path above
                        cp_item<true, false>(st, in, itl, nullptr, 0, 0, sink);
                    } else {
                        if (q == 0) cp_item<false, true>(st, in, itl, nxt, nx.hp, nx.map_elems, sink);
                        else cp_item<false, false>(st, in, itl, nxt, nx.hp, nx.map_elems, sink);
                    }
                }
                __syncthreads();
            }
        }
    } else if (FUSED == 1) {
        // ---- fused front end: two warps per image --------------------------------------------------------------
        int* bufs = reinterpret_cast<int*>(tile + SN_TB * pitch);
        const int n_img = tid >> 6, lt = tid & 63;
        const int sample = s0 + n_img;
        const bool live = sample < B;
        int* buf0 = bufs + (size_t)n_img * 2 * fr.max_elems;
        int* buf1 = buf0 + fr.max_elems;
        double* trow = tile + (size_t)n_img * pitch;
        if (live) {
            const size_t src = source_image(fr.bi, (size_t)sample);
            if (lt == 0) {
                const long long lab = fr.bi.cursor ? fr.bi.labels_all[src] : (labels ? labels[sample] : 0);
                s_label[n_img] = lab;
                if (fr.bi.labels_batch) fr.bi.labels_batch[sample] = lab;
            }
            load_image<uint8_t, int>(fr.images + image_slot(fr.bi, src) * fr.H * fr.W, buf0, fr.H, fr.W, lt, 64);
        } else {
            for (int i = lt; i < pitch; i += 64) trow[i] = 0.0;
            if (lt == 0) s_label[n_img] = -1;
        }
        __syncthreads();
        int* cur = buf0;
        int* nxt = buf1;
        for (int s = 0; s < fr.stages.n; ++s) {
            const Stage& st = fr.stages.s[s];
            if (live) {
                if (s == fr.stages.n - 1) {
                    EmitTile<!INFER> e{trow, INFER ? nullptr : feats + (size_t)sample * L, st.h_out, st.h_out * st.w_out, fr.sc};
                    run_stage<int>(st, cur, e, lt, 64);
                } else {
                    EmitMaps<int> e{nxt, st.h_out, st.h_out * st.w_out};
                    run_stage<int>(st, cur, e, lt, 64);
                }
            }
            __syncthreads();
            int* tmp = cur; cur = nxt; nxt = tmp;
        }
    } else {
        if (tid < SN_TB) s_label[tid] = (labels && s0 + tid < B) ? labels[s0 + tid] : -1;
    }

    if (PREWAIT) {   // everything above ran under the previous step's exchange kernel (prewait 1) or under the tail of its
                     // weight-gradient kernel (prewait 2); the parameters are final from here on
        asm volatile("griddepcontrol.wait;" ::: "memory");
        load_params();
        if (FUSED == 2 && fr.prewait == 2) {
            // the previous step's kernel B was still reading the feature buffer until now: this tile's rows go out from shared memory
            const int n_live = min(SN_TB, B - s0);
            for (int gi = 0; gi < n_live; ++gi) {
                double* __restrict__ dst = feats + (size_t)(s0 + gi) * L;
                const double* src = tile + (size_t)gi * pitch;
                for (int k = tid; k < L; k += SNA_THREADS) dst[k] = src[k];
            }
        }
    }
    SN_PHASE(3);
    // ---- layer 0: z = W0 a0 on DMMA, K split across the 16 warps ----------------------------------------------------
    // The first U k-steps of this warp's W0 fragments were loaded into registers at the very top (w_pre), the rest of
    // its K range was prefetched into L1: the L2 round trips overlap the front end instead of following it.
    {
        double acc[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0;
        const int sample = s0 + g;
        const bool sample_ok = sample < B;
        const double* __restrict__ frow = feats + (size_t)(sample_ok ? sample : 0) * L;
        const double* trow = tile + (size_t)g * pitch;
        {
            double bf[SN_U];
#pragma unroll
            for (int u = 0; u < SN_U; ++u) {
                const int k = (ks_begin + u) * 4 + t;
                const bool kok = (ks_begin + u) < ks_end && k < L;
                if (FUSED) bf[u] = kok ? trow[k] : 0.0;                                        // B frag: row t (k), col g (sample)
                else bf[u] = (kok && sample_ok) ? __ldg(frow + k) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < SN_U; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < mf) sn_dmma(acc[i][0], acc[i][1], w_pre[u][i], bf[u]);
        }
        for (int ks = ks_begin + SN_U; ks < ks_end; ks += SN_U) {
            double af[SN_U][4], bf[SN_U];
#pragma unroll
            for (int u = 0; u < SN_U; ++u) {
                const int k = (ks + u) * 4 + t;
                const bool kok = (ks + u) < ks_end && k < L;
                const double* wp = W0 + (size_t)k * R0 + g;
#pragma unroll
                for (int i = 0; i < 4; ++i) af[u][i] = (kok && rowok[i]) ? sn_ld<PREWAIT ? 2 : 0>(wp + i * 8) : 0.0;  // A frag: row g (m), col t (k)
                if (FUSED) bf[u] = kok ? trow[k] : 0.0;
                else bf[u] = (kok && sample_ok) ? __ldg(frow + k) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < SN_U; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < mf) sn_dmma(acc[i][0], acc[i][1], af[u][i], bf[u]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // C frag: row g (m), cols 2t, 2t+1 (sample); [warp][sample][36]: conflict-free both ways
            zpart[(warp * SN_TB + 2 * t) * SN_ZPITCH + i * 8 + g] = acc[i][0];
            zpart[(warp * SN_TB + 2 * t + 1) * SN_ZPITCH + i * 8 + g] = acc[i][1];
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");   // this thread's share of the small parameters has landed
    __syncthreads();
    SN_PHASE(4);
    const int last = d.n_layers - 1;
    const int RL = d.rows[last];
    // ---- narrow part: warp n owns sample n from here to its deltas (lane = neuron), so the layers only need warp-level
    // synchronisation; warps 8..15 rejoin for the gradient partials.
    if (warp < SN_TB) {
        const int n = warp;           // sample within the tile
        const int m = lane;           // neuron
        const int sample = s0 + n;
        const bool live = sample < B;
        {
            double zp[SNA_WARPS];
#pragma unroll
            for (int w = 0; w < SNA_WARPS; ++w) zp[w] = zpart[(w * SN_TB + n) * SN_ZPITCH + m];
#pragma unroll
            for (int o = 1; o < SNA_WARPS; o <<= 1)      // fixed pairwise tree over the 16 K-splits
#pragma unroll
                for (int w = 0; w < SNA_WARPS; w += 2 * o) zp[w] += zp[w + o];
            SN_PHASE(16);
            if (m < R0) {
                const double z = zp[0] + s_small[m];            // w * a + b      (rcn.rs:287)
                s_act[0][n][m] = sn_sigmoid(z);                 // sigmoid(&z)    (rcn.rs:289)
            }
        }
        SN_PHASE(17);
        __syncwarp();
        // ---- narrow layers.  Every layer loop below is unrolled over kSmallNetMaxLayers with a guard, so the descriptor
        // fields (rows / offsets) are read with STATIC constant-bank offsets -- an operand of the instruction -- instead of a
        // dependent LDC per use, and the k loops run on four independent FMA chains ------------------------------------
#pragma unroll
        for (int l = 1; l < kSmallNetMaxLayers; ++l) {
            if (l < d.n_layers) {
                const int R = d.rows[l], C = d.rows[l - 1];
                if (m < R) {
                    const double* W = s_small + (d.w_off[l] - small_base) + m;
                    const double* av = &s_act[l - 1][n][0];
                    double z0 = 0.0, z1 = 0.0, z2 = 0.0, z3 = 0.0;
                    int k = 0;
#pragma unroll 2
                    for (; k + 3 < C; k += 4) {
                        z0 = fma(W[k * R], av[k], z0);
                        z1 = fma(W[(k + 1) * R], av[k + 1], z1);
                        z2 = fma(W[(k + 2) * R], av[k + 2], z2);
                        z3 = fma(W[(k + 3) * R], av[k + 3], z3);
                    }
                    for (; k < C; ++k) z0 = fma(W[k * R], av[k], z0);
                    const double z = ((z0 + z1) + (z2 + z3)) + s_small[d.b_off[l] - small_base + m];
                    s_act[l][n][m] = sn_sigmoid(z);
                }
                __syncwarp();
            }
        }
        SN_PHASE(5);
        // ---- activations out ---------------------------------------------------------------------------------------
        if constexpr (!INFER) {
            int off = 0;
#pragma unroll
            for (int l = 0; l < kSmallNetMaxLayers; ++l) {
                if (l < d.n_layers) {
                    const int R = d.rows[l];
                    if (live && m < R) acts[(size_t)off * B + (size_t)sample * R + m] = s_act[l][n][m];
                    off += R;
                }
            }
        }
        SN_PHASE(18);
        if (INFER || backward) {
            // ---- output delta (rcn.rs:299) and batch statistics (rcn.rs:152-157) ---------------------------------------
            const bool out = m < RL;
            double y = 0.0;
            if (out && live) y = onehot ? onehot[(size_t)sample * RL + m] : ((s_label[n] == (long long)m) ? 1.0 : 0.0);
            const double a = out ? s_act[last][n][m] : 0.0;
            if constexpr (!INFER) {
                if (out) s_del[last][n][m] = (a - y) * (a * (1.0 - a));
            }
            {
                double mx = out ? a : -1.0;                        // activations are in (0, 1)
                const double df = a - y;                           // 0 for lanes beyond the output layer
                double cost = out ? df * df : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {                 // both butterflies in one pass: fixed order, deterministic
                    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                    cost += __shfl_xor_sync(0xffffffffu, cost, o);
                }
                const bool ok = __all_sync(0xffffffffu, !out || (((a == mx) ? 1.0 : 0.0) == y));
                if (m == 0) {
                    s_cost[n] = live ? cost * 0.5 : 0.0;
                    s_hit[n] = (live && ok) ? 1ull : 0ull;
                }
            }
            if constexpr (INFER) {
                // the class label with argmax_last_kernel's sequential scan: last maximal element wins (rcn.rs:92-97), and a
                // NaN output gives the label classify gives
                if (inf.labels_out && live && m == 0) {
                    int best = 0;
                    double bv = s_act[last][n][0];
                    for (int i = 1; i < RL; ++i) {
                        const double v = s_act[last][n][i];
                        if (!(v < bv)) { bv = v; best = i; }
                    }
                    inf.labels_out[sample] = best;
                }
            } else {
            SN_PHASE(19);
            __syncwarp();
            // ---- backward-data chain (rcn.rs:305-309) -------------------------------------------------------------------
#pragma unroll
            for (int l = kSmallNetMaxLayers - 2; l >= 0; --l) {
                if (l < last) {
                    const int R = d.rows[l], Ru = d.rows[l + 1];
                    if (m < R) {
                        const double* Wu = s_small + (d.w_off[l + 1] - small_base) + m * Ru;  // Ru x R column-major: (k, m) at m*Ru + k
                        const double* dv = &s_del[l + 1][n][0];
                        double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
                        int k = 0;
#pragma unroll 2
                        for (; k + 3 < Ru; k += 4) {
                            v0 = fma(Wu[k], dv[k], v0);
                            v1 = fma(Wu[k + 1], dv[k + 1], v1);
                            v2 = fma(Wu[k + 2], dv[k + 2], v2);
                            v3 = fma(Wu[k + 3], dv[k + 3], v3);
                        }
                        for (; k < Ru; ++k) v0 = fma(Wu[k], dv[k], v0);
                        const double al = s_act[l][n][m];
                        s_del[l][n][m] = ((v0 + v1) + (v2 + v3)) * (al * (1.0 - al));
                    }
                    __syncwarp();
                }
            }
            SN_PHASE(20);
            int off = 0;
#pragma unroll
            for (int l = 0; l < kSmallNetMaxLayers; ++l) {
                if (l < d.n_layers) {
                    const int R = d.rows[l];
                    if (live && m < R) deltas[(size_t)off * B + (size_t)sample * R + m] = s_del[l][n][m];
                    off += R;
                }
            }
            }   // !INFER
        }
    }
    SN_PHASE(21);
    if (!INFER && !backward) { RCN_TL_END(d.tl, 0); return; }
    __syncthreads();
    SN_PHASE(6);
    if (tid == SNA_THREADS - 32) {
        double c = 0.0;
        unsigned long long h = 0;
#pragma unroll
        for (int i = 0; i < SN_TB; ++i) { c += s_cost[i]; h += s_hit[i]; }
        stats_partial[2 * tile_idx] = c;
        reinterpret_cast<unsigned long long*>(stats_partial)[2 * tile_idx + 1] = h;
    }
    if constexpr (INFER) {
        // ---- the last CTA to finish (ticket after a fence, as batch_stats_kernel) adds the partials in exactly the order of
        // kernel B's statistics CTA: same partials, same order, so the result is bit-identical to the training step's
        // {cost, hits} on the same batch.  It resets the ticket, so a captured launch can be replayed.
        __shared__ bool s_last;
        if (tid == SNA_THREADS - 32) {
            __threadfence();
            const unsigned t = atomicAdd(inf.ticket, 1u);
            s_last = (t == gridDim.x - 1);
            if (s_last) *inf.ticket = 0;
        }
        __syncthreads();
        if (s_last) {   // uniform across the CTA
            const int n_stat = (int)gridDim.x;
            const int per_l = (n_stat + 31) / 32;
            // Lane l of warp 0 adds partials l*per_l, l*per_l + 1, ... in order.  Up to SN_RJ partials per lane it loads them
            // itself; above that (B > 16 384) the loads are not left to one warp, a chain of dependent L2 round trips that
            // grows with B: all 16 warps stage SN_RJ consecutive partials of every lane's range into shared memory (the layer-0
            // partial-sum area, free by now) and warp 0 folds them, in the same order.  Measured with profiles/eval_bench.py on
            // B200s at 1000 W (separate runs), staging at every size against the warp-0 loop: 9.42 against 9.53 ms at
            // B = 1 048 576, equal at 10 000, 16.4 against 14.4 us at B = 1.
            constexpr int SN_RJ = 64, SN_RPITCH = SN_RJ + 1;       // odd pitch: lane l's row starts in bank 2l mod 32
            double c = 0.0;
            unsigned long long h = 0;
            if (per_l <= SN_RJ) {
                if (warp != 0) return;
                __threadfence();
                for (int i = lane * per_l; i < min(n_stat, (lane + 1) * per_l); ++i) {
                    c += __ldcg(stats_partial + 2 * i);
                    h += __ldcg(reinterpret_cast<const unsigned long long*>(stats_partial) + 2 * i + 1);
                }
            } else {
                __threadfence();
                double* rc = zpart;
                unsigned long long* rh = reinterpret_cast<unsigned long long*>(zpart + 32 * SN_RPITCH);
                for (int j0 = 0; j0 < per_l; j0 += SN_RJ) {
                    for (int e = tid; e < 32 * SN_RJ; e += SNA_THREADS) {
                        const int l = e / SN_RJ, jj = e - l * SN_RJ;
                        const int i = l * per_l + j0 + jj;
                        if (j0 + jj < per_l && i < n_stat) {
                            rc[l * SN_RPITCH + jj] = __ldcg(stats_partial + 2 * i);
                            rh[l * SN_RPITCH + jj] = __ldcg(reinterpret_cast<const unsigned long long*>(stats_partial) + 2 * i + 1);
                        }
                    }
                    __syncthreads();
                    if (warp == 0) {
                        const int n_j = min(SN_RJ, min(per_l, n_stat - lane * per_l) - j0);
                        for (int jj = 0; jj < n_j; ++jj) {
                            c += rc[lane * SN_RPITCH + jj];
                            h += rh[lane * SN_RPITCH + jj];
                        }
                    }
                    __syncthreads();
                }
                if (warp != 0) return;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                c += __shfl_down_sync(0xffffffffu, c, o);
                h += __shfl_down_sync(0xffffffffu, h, o);
            }
            if (lane == 0) {
                if (inf.accumulate) {   // chunks in order: ((c0 + c1) + c2) ...
                    c = inf.stats[0] + c;
                    h += reinterpret_cast<const unsigned long long*>(inf.stats)[1];
                }
                inf.stats[0] = c;
                reinterpret_cast<unsigned long long*>(inf.stats)[1] = h;
            }
        }
        return;
    }
    // ---- epoch mode: ask L2 for the images this tile will load in the NEXT step (same tile index, cursor advanced like the
    // update does, rcn.rs:147): 20 us from now their bulk loads hit L2 instead of paying an HBM round trip at the head of
    // the step's critical path.  Nobody waits for these requests.
    if (FUSED == 2 && warp == 1 && lane < SN_TB && fr.bi.cursor && !fr.bi.window && fr.bi.batch > 0 && s0 + lane < B) {
        long long nx = __ldcg(fr.bi.cursor) + fr.bi.batch;
        if (nx + fr.bi.batch > fr.bi.n_samples) nx = 0;
        const long long pos = nx + s0 + lane;
        const size_t src = (size_t)(fr.bi.perm ? fr.bi.perm[pos] : pos);
        const uint32_t img_bytes = (uint32_t)(fr.H * fr.W);
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(fr.images + src * img_bytes), "r"(img_bytes) : "memory");
    }
    SN_PHASE(7);
    RCN_TL_END(d.tl, 0);
}

template <int FUSED, bool PREWAIT>
__global__ void __launch_bounds__(SNA_THREADS, 1)
smallnet_fwd_bwd_kernel(const __grid_constant__ SmallNetDesc d, const double* __restrict__ params,
                        double* __restrict__ feats, int B, const double* __restrict__ onehot,
                        const int64_t* __restrict__ labels, double* __restrict__ acts, double* __restrict__ deltas,
                        double* __restrict__ stats_partial, int backward, const __grid_constant__ SmallNetFront fr) {
    extern __shared__ __align__(128) unsigned char sn_smem[];
    sn_phase_a<FUSED, PREWAIT, false>(d, params, feats, B, onehot, labels, acts, deltas, stats_partial, backward, fr,
                                      (int)blockIdx.x, sn_smem, SnInfer{});
}

// Inference variant of kernel A (test-set evaluation): the same front end and forward pass per tile of 8 samples, then the
// cost and hit rule of the training epilogue, the optional argmax labels, and one {cost, hits} for the whole launch.
// FUSED 1 / 2: the features are computed from `fr.images` and stay in shared memory.
template <int FUSED>
__global__ void __launch_bounds__(SNA_THREADS, 1)
smallnet_infer_kernel(const __grid_constant__ SmallNetDesc d, const double* __restrict__ params, int B,
                      const int64_t* __restrict__ labels, double* __restrict__ stats_partial, const __grid_constant__ SnInfer inf,
                      const __grid_constant__ SmallNetFront fr) {
    static_assert(FUSED == 1 || FUSED == 2, "the inference kernel runs the fused front end");
    extern __shared__ __align__(128) unsigned char sn_smem[];
    sn_phase_a<FUSED, false, true>(d, params, nullptr, B, nullptr, labels, nullptr, nullptr, stats_partial, 0,
                                   fr, (int)blockIdx.x, sn_smem, inf);
}

// ------------------------------------------------------------------------------------------------
// Kernel B: dW/db.  grid = (col_groups + small_groups, S) launched as thread-block CLUSTERS of (1, S, 1): the S CTAs of a
// cluster own the same 64 columns of dW0 (or, for blockIdx.x >= col_groups, a share of db0 + the narrow layers) and one K-split
// of the batch each.  Every CTA leaves its partial tile in its own shared memory; after a cluster barrier each rank
// sums 1/S of the tile over all S ranks through distributed shared memory, in rank order (deterministic), and
// writes the flat gradient buffer.  No partials ever touch L2/HBM.
// ------------------------------------------------------------------------------------------------
constexpr int SNB_TILE = 32 * 64;   // padded partial tile: 32 rows x 64 columns

// MODE 0: gradients only.  MODE 1: also push the final values into the data-parallel peers' receive slots (dp.cu
// protocol; the update kernel then only receives).  MODE 2: single GPU, apply the SGD update to the finished elements
// right here (SnUpdate).
// Whatever the mode, when `upd.cursor` is set the statistics thread also advances the epoch cursor and writes the per-step
// result ring (on a data-parallel group that makes the cursor final BEFORE the exchange kernel runs, which is what lets the
// next step's kernel A read it ahead of its griddepcontrol.wait).
// (Measured and dropped, round 2: 48 columns per CTA = 17 column groups x 8 K-splits + 8 = 144 CTAs "one per SM" ran 11.2 us
// instead of 6.1 -- B200 co-schedules only ~15 clusters of 8 CTAs, so 18 clusters take two waves.)
// Each column CTA owns 64 columns of dW0, one warp per 8 columns.
template <int MODE>
__device__ __forceinline__ void sn_phase_b(const SmallNetDesc& d, const double* __restrict__ feats,
                                           const double* __restrict__ acts, const double* __restrict__ deltas,
                                           int B, int ksplit, int col_groups, double* __restrict__ grads,
                                           const double* __restrict__ stats_partial, int n_stat, double* __restrict__ stats,
                                           const DpPush& dp, const SnUpdate& upd, const int chunk /* samples per staging pass of the small CTA */,
                                           const int cg_idx, const int rank, const int S,
                                           double* sP, double* sD /* [2][64 * SN_DPITCH]: double-buffered 64-sample delta_0 chunk */,
                                           const long long cur0_early /* >= 0: the cursor was advanced at the top */) {
    constexpr bool DP = MODE == 1;
    constexpr bool UPD = MODE == 2;
    constexpr int CW = 64;                                   // columns of dW0 per CTA
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    RCN_TL_BEGIN(d.tl, 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int L = d.n_in, R0 = d.rows[0];
    const int b_begin = rank * ksplit;
    const int b_end = min(B, b_begin + ksplit);
    const bool is_col = cg_idx < col_groups;
    // the "small" parameter block b0|W1|b1|... is dealt to the (gridDim.x - col_groups) small column groups in contiguous halves
    const int small_groups = (int)gridDim.x - col_groups;
    const int e_per = (d.n_params - d.b_off[0] + small_groups - 1) / small_groups;
    const int e_lo = is_col ? 0 : (cg_idx - col_groups) * e_per;
    const int e_hi = is_col ? 0 : min(d.n_params - d.b_off[0], e_lo + e_per);
    const int small_base = d.b_off[0];
    const int n_small = d.n_params - small_base;

    if (is_col) {
        const int mf = (R0 + 7) >> 3;
        constexpr int NWC = CW / 8;                          // warps across the columns
        constexpr int KQ = 8 / NWC;                          // warps sharing a column octet (each 64 / KQ samples of a chunk)
        const int oct = warp % NWC, kq = warp / NWC;
        const int col = cg_idx * CW + oct * 8 + g;          // B frag column (feature index)
        const bool col_ok = col < L;
        constexpr int U = 16 / KQ;                           // k-steps per warp per 64-sample chunk
        double acc[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0;
        // Chunks are taken in PAIRS: both chunks' A0 fragments (2 x U loads per lane) and both delta slices are requested
        // before the one barrier, so a K-split of 128 samples (the canonical case) pays ONE L2 round trip, not two.
        auto load_feats = [&](double (&bf)[U], int c0) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int b = c0 + kq * (64 / KQ) + u * 4 + t;
                bf[u] = (b < b_end && col_ok) ? feats[(size_t)b * L + col] : 0.0;   // B frag: row t (sample), col g (feature)
            }
        };
        auto load_delta = [&](double (&vd)[8], int c0) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {            // 64 x 32 slice = 8 elements per thread
                const int idx = u * SNB_THREADS + tid;
                const int kk = idx >> 5, mm = idx & 31;
                const int b = c0 + kk;
                vd[u] = (mm < R0 && b < b_end) ? deltas[(size_t)b * R0 + mm] : 0.0;
            }
        };
        auto store_delta = [&](const double (&vd)[8], double* sd) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int idx = u * SNB_THREADS + tid;
                sd[(idx >> 5) * SN_DPITCH + (idx & 31)] = vd[u];
            }
        };
        auto mma_chunk = [&](const double (&bf)[U], const double* sd) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int kk = kq * (64 / KQ) + u * 4 + t;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < mf) sn_dmma(acc[i][0], acc[i][1], sd[kk * SN_DPITCH + i * 8 + g], bf[u]);  // A frag: row g (m), col t
            }
        };
        for (int c0 = b_begin; c0 < b_end; c0 += 128) {
            const bool two = c0 + 64 < b_end;
            double bf0[U], bf1[U], vd0[8], vd1[8];
            load_feats(bf0, c0);
            load_delta(vd0, c0);
            if (two) { load_feats(bf1, c0 + 64); load_delta(vd1, c0 + 64); }
            store_delta(vd0, sD);
            if (two) store_delta(vd1, sD + 64 * SN_DPITCH);
            __syncthreads();   // both slices staged
            mma_chunk(bf0, sD);
            if (two) mma_chunk(bf1, sD + 64 * SN_DPITCH);
            if (c0 + 128 < b_end) __syncthreads();   // before the slices are overwritten
        }
        const int cl = kq * CW + oct * 8 + 2 * t;           // C frag: row g (m), cols 2t, 2t+1; one CW x 32 tile per kq
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            sP[cl * 32 + i * 8 + g] = acc[i][0];
            sP[(cl + 1) * 32 + i * 8 + g] = acc[i][1];
        }
    } else {
        // ---- db_l (all layers) and dW_l = sum_b delta_l a_{l-1}^T (narrow layers, rcn.rs:302-303,309-310) for this K-split:
        // the split's activations (layers 0 .. n-2) and deltas (all layers) are staged in shared memory chunk by chunk --
        // per layer one contiguous, coalesced block [sample][rows_l], exactly as it lies in global memory -- and every
        // thread owns the entries o = tid, tid + 256, ... of the "small" parameter block b0|W1|b1|..., adding the samples in
        // index order on two interleaved chains (even / odd samples; deterministic).  This CTA would otherwise idle while
        // the column CTAs run their DMMAs, and kernel A no longer spends its tail on per-tile partial sums.
        double* stg = sP + ((n_small + 1) & ~1);                 // staging area behind the partial tile (dynamic smem)
        int per_sample = 0;                                       // doubles per sample in a chunk: a_0..a_{n-2} | delta_0..delta_{n-1}
        for (int l = 0; l + 1 < d.n_layers; ++l) per_sample += d.rows[l];
        const int act_doubles = per_sample;
        for (int l = 0; l < d.n_layers; ++l) per_sample += d.rows[l];
        for (int o = tid; o < e_hi - e_lo; o += SNB_THREADS) sP[o] = 0.0;
        for (int c0 = b_begin; c0 < b_end; c0 += chunk) {
            const int cn = min(chunk, b_end - c0);
            __syncthreads();                                      // sP zeroed / the previous chunk consumed
            {   // asynchronous copies: no register dependency, every request of the chunk is in flight at once (one L2 round trip)
                auto stage = [&](const double* src, int n, int soff) {
                    for (int i = tid; i < n; i += SNB_THREADS) {
                        const unsigned dst = (unsigned)__cvta_generic_to_shared(stg + soff + i);
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src + i) : "memory");
                    }
                };
                size_t goff = 0;
                int soff = 0;
                for (int l = 0; l + 1 < d.n_layers; ++l) {        // activations of layers 0 .. n-2
                    const int R = d.rows[l];
                    stage(acts + goff * B + (size_t)c0 * R, cn * R, soff);
                    goff += R; soff += chunk * R;
                }
                goff = 0;
                for (int l = 0; l < d.n_layers; ++l) {            // deltas of every layer
                    const int R = d.rows[l];
                    stage(deltas + goff * B + (size_t)c0 * R, cn * R, soff);
                    goff += R; soff += chunk * R;
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_all;" ::: "memory");
            }
            __syncthreads();
            for (int o = e_lo + tid; o < e_hi; o += SNB_THREADS) {
                // decode o -> layer l, row m, and (for a weight entry) column k
                int a_blk = 0, d_blk = act_doubles;               // per-sample offsets of a_{l-1} / delta_l
                const double* dp_ = nullptr;
                const double* ap_ = nullptr;
                int dR = 0, aR = 0;
                for (int l = 0; l < d.n_layers; ++l) {
                    const int R = d.rows[l];
                    const int bo = d.b_off[l] - small_base;
                    if (o >= bo && o < bo + R) { dp_ = stg + d_blk * chunk + (o - bo); dR = R; break; }
                    if (l >= 1) {
                        const int C = d.rows[l - 1];
                        const int wo = d.w_off[l] - small_base;
                        if (o >= wo && o < wo + R * C) {
                            const int k = (o - wo) / R, m = (o - wo) - k * R;
                            dp_ = stg + d_blk * chunk + m; dR = R;
                            ap_ = stg + a_blk * chunk + k; aR = C;
                            break;
                        }
                        a_blk += C;
                    }
                    d_blk += R;
                }
                if (!dp_) continue;
                double s0 = 0.0, s1 = 0.0;
                int b = 0;
                if (ap_) {
#pragma unroll 4
                    for (; b + 1 < cn; b += 2) {                  // 16 shared loads in flight per thread
                        s0 = fma(dp_[b * dR], ap_[b * aR], s0);
                        s1 = fma(dp_[(b + 1) * dR], ap_[(b + 1) * aR], s1);
                    }
                    if (b < cn) s0 = fma(dp_[b * dR], ap_[b * aR], s0);
                } else {
#pragma unroll 4
                    for (; b + 1 < cn; b += 2) { s0 += dp_[b * dR]; s1 += dp_[(b + 1) * dR]; }
                    if (b < cn) s0 += dp_[b * dR];
                }
                sP[o - e_lo] += s0 + s1;
            }
        }
    }

    // ---- cross-split reduction through distributed shared memory, rank order ----------------------------------------
    cluster.sync();
    const int n_out = is_col ? CW * 32 : e_hi - e_lo;
    const int per = (n_out + S - 1) / S;
    const int o_lo = rank * per, o_hi = min(n_out, o_lo + per);
    // data-parallel group: the final values also go straight into the peers' receive slots (dp.cu protocol), so the
    // exchange overlaps this kernel's tail and the launch of the update kernel
    const size_t dp_par = DP ? dp_push_parity_offset(dp) : 0;
    for (int o = o_lo + tid; o < o_hi; o += SNB_THREADS) {
        // destination first: the old parameter value (fused update) is in flight while the peers' partials are read
        long long gi = -1;
        if (is_col) {
            const int m = o & 31, col = cg_idx * CW + (o >> 5);
            if (m < R0 && col < L) gi = d.w_off[0] + (long long)col * R0 + m;
        } else {
            gi = small_base + e_lo + o;
        }
        double pold = 0.0;
        if (UPD && gi >= 0) pold = upd.params[gi];
        // all S remote reads are issued before the first add (one DSMEM round trip, not S dependent ones; S <= 8)
        double rv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            rv[q] = 0.0;
            if (q < S) rv[q] = cluster.map_shared_rank(sP, q)[o];
        }
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (q < S) s += rv[q];
        if (gi >= 0) {
            if (DP) dp_push_value(dp, dp_par, (size_t)gi, s);
            grads[gi] = s;
            if (UPD) upd.params[gi] = sgd_apply(pold, upd.scale, s);
        }
    }
    if (!is_col && cg_idx == col_groups && rank == 0 && tid < 32 && stats) {
        // 32 lanes, each a contiguous chunk in order, then a fixed-order shuffle tree => deterministic
        const int per_l = (n_stat + 31) / 32;
        double c = 0.0;
        unsigned long long h = 0;
        for (int i = tid * per_l; i < min(n_stat, (tid + 1) * per_l); ++i) {
            c += stats_partial[2 * i];
            h += reinterpret_cast<const unsigned long long*>(stats_partial)[2 * i + 1];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c += __shfl_down_sync(0xffffffffu, c, o);
            h += __shfl_down_sync(0xffffffffu, h, o);
        }
        if (tid == 0) {
            stats[0] = c;
            reinterpret_cast<unsigned long long*>(stats)[1] = h;
            if (upd.cursor) {   // what sgd_update_kernel does on the side (kernel A of this step is long done)
                const long long cur0 = cur0_early >= 0 ? cur0_early : *upd.cursor;
                if (upd.stats_ring) {
                    double* dst = upd.stats_ring + 2 * (cur0 / upd.batch);
                    dst[0] = c;
                    reinterpret_cast<unsigned long long*>(dst)[1] = h;
                }
                if (cur0_early < 0) {
                    long long cur = cur0 + upd.batch;   // next chunk of chunks_exact(batch) (rcn.rs:147), remainder dropped
                    if (cur + upd.batch > upd.n_samples) cur = 0;
                    *upd.cursor = cur;
                }
            }
        }
    }
    // nobody leaves while a peer may still read its tile.  RELAXED arrive: this barrier orders no memory (a peer arrives after
    // it has consumed the values it read from my tile), so it must not wait for this CTA's global stores to drain the way
    // the release fence of cluster.sync() does (ncu: 9 % of the kernel's samples sat in that membar).
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
    RCN_TL_END(d.tl, 1);
}

template <int MODE>
__global__ void __launch_bounds__(SNB_THREADS) smallnet_wgrad_kernel(const __grid_constant__ SmallNetDesc d,
                                                                     const double* __restrict__ feats,
                                                                     const double* __restrict__ acts,
                                                                     const double* __restrict__ deltas, int B, int ksplit,
                                                                     int col_groups, double* __restrict__ grads,
                                                                     const double* __restrict__ stats_partial, int n_stat,
                                                                     double* __restrict__ stats, const __grid_constant__ DpPush dp,
                                                                     const __grid_constant__ SnUpdate upd, int chunk) {
    extern __shared__ __align__(16) double sP_dyn[];          // partial tile: SNB_TILE (col CTAs) or n_small doubles + the small CTA's staging area
    __shared__ __align__(16) double sD_static[2 * 64 * SN_DPITCH];   // 36 KB
    // grid (col_groups + 1, S) in clusters of (1, S, 1): blockIdx.y == cluster.block_rank()
    // Early trigger (the successor's CTAs are scheduled under this kernel and wait in griddepcontrol.wait): on one GPU, and on
    // a data-parallel group when this kernel pushed to the peers (MODE 1) -- its successor is then the exchange kernel, which
    // waits for this kernel's completion before it lets the next kernel A start.  Not in the other group modes: their
    // successor may be a PREWAIT kernel A, whose early part overwrites the feature buffer this kernel reads.
    //
    // One GPU with a device-side cursor: the next kernel A may read the cursor BEFORE its own griddepcontrol.wait (prewait 2: its
    // front end runs under this kernel's tail), so the cursor is advanced before this kernel lets it start -- the statistics CTA
    // first waits for this step's kernel A (the cursor's last reader), advances the cursor, and only then triggers; the launch
    // of the dependents needs every CTA's trigger, so it cannot overtake that store.
    long long cur0_early = -1;
    if (dp.world <= 1 && upd.cursor && upd.early_cursor && blockIdx.x == (unsigned)col_groups && blockIdx.y == 0) {
        __shared__ long long s_cur0;
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (threadIdx.x == 0) {
            const long long c0 = *upd.cursor;
            long long cur = c0 + upd.batch;   // next chunk of chunks_exact(batch) (rcn.rs:147), remainder dropped
            if (cur + upd.batch > upd.n_samples) cur = 0;
            *upd.cursor = cur;
            s_cur0 = c0;
            __threadfence();
        }
        __syncthreads();
        cur0_early = s_cur0;
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    } else {
        if (dp.world <= 1 || MODE == 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    sn_phase_b<MODE>(d, feats, acts, deltas, B, ksplit, col_groups, grads, stats_partial, n_stat, stats, dp, upd, chunk,
                     (int)blockIdx.x, (int)blockIdx.y, (int)gridDim.y, sP_dyn, sD_static, cur0_early);
}

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------
bool smallnet_eligible(const SmallNetDesc& d) {
    if (d.n_layers < 1 || d.n_layers > kSmallNetMaxLayers) return false;
    for (int l = 0; l < d.n_layers; ++l)
        if (d.rows[l] < 1 || d.rows[l] > 32) return false;
    return d.n_in >= 1;
}

// K-splits of the batch = cluster size of kernel B (portable maximum 8), each a whole number of 64-sample chunks.
static void smallnet_splits(size_t B, int* splits, int* ksplit) {
    int s = 1;
    while (s < 8 && (size_t)s * 64 < B) s *= 2;
    size_t ks = (B + s - 1) / s;
    ks = (ks + 63) / 64 * 64;
    *splits = (int)((B + ks - 1) / ks);
    if (*splits < 1) *splits = 1;
    *ksplit = (int)ks;
}

size_t smallnet_max_batch() { return (size_t)1 << 22; }

// Highest launch priority for the training kernels: pending CTAs of kernels A / B win the SMs (kernel A needs a whole SM
// per CTA) against lower-priority work queued on the same device.  (It was added against the SM-issued prefetch kernel of
// the host-dataset loop, which no longer exists; whether it still pays has not been measured.)
static int sn_high_priority() {
    static const int prio = []() {
        int least = 0, greatest = 0;
        if (cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) { cudaGetLastError(); return 0; }
        return greatest;
    }();
    return prio;
}

static size_t kernel_a_smem(const SmallNetDesc& d, const SmallNetFront* fr) {
    size_t bytes = ((size_t)SNA_WARPS * SN_TB * SN_ZPITCH + SN_MAX_SMALL) * sizeof(double);
    if (fr) {
        bytes += (size_t)SN_TB * (d.n_in + SN_TILE_PAD) * sizeof(double);
        if (fr->use_cp) bytes += 128 + (size_t)SN_TB * (size_t)fr->cp.stage_bytes +
                                 (size_t)(fr->cp_pairs ? SN_TB / 2 : SN_TB) * (size_t)fr->cp.tile_ints * sizeof(int);
        else bytes += (size_t)SN_TB * 2 * fr->max_elems * sizeof(int);
    }
    return bytes;
}

bool smallnet_front_fits(const SmallNetDesc& d, const SmallNetFront& fr) { return kernel_a_smem(d, &fr) <= 200 * 1024; }

void smallnet_front_select(const FeaturePlan& plan, SmallNetFront* fr) {
    static const bool off = []() { const char* e = getenv("RCN_CUDA_FEATURES_STAGED"); return e && e[0] == '0'; }();
    fr->use_cp = 0;
    fr->cp_pairs = 0;
    if (off || (reinterpret_cast<uintptr_t>(fr->images) & 15) != 0 || ((size_t)fr->H * fr->W) % 16 != 0) return;
    if (!make_cp_plan(plan, (size_t)fr->H, (size_t)fr->W, &fr->cp)) return;
    fr->use_cp = 1;
    long long bound = 255;   // largest magnitude of an intermediate after the plan's stages
    for (int q = 0; q < fr->cp.n; ++q) bound *= 4;
    fr->cp_pairs = bound <= 2048;   // one stage (1020; two reach 4080): the form cp_item_pair and kernel A's int32 loop assume
}

static int launch_kernel_a(const SmallNetDesc& d, const double* params, double* feats, size_t B, const double* onehot,
                           const int64_t* labels, double* acts, double* deltas, double* stats_partial,
                           int backward, const SmallNetFront* fr, cudaStream_t stream) {
    const unsigned n_tiles = cdiv(B, SN_TB);
    const size_t smem = kernel_a_smem(d, fr);
    static SmallNetFront empty_front{};
    const int Bi = (int)B;
    auto launch = [&](auto kern, SmemAttrCache& attr, const char* name, const SmallNetFront& front) -> int {
        // (Measured and dropped, round 2: asking for the all-shared L1 split on every step kernel -- so that no SM is
        // reconfigured at a kernel boundary -- made the step 0.6 us SLOWER: kernel A's tail of W0 is prefetched into L1.)
        if (attr.need(smem)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(n_tiles, 1, 1);
        cfg.blockDim = dim3(SNA_THREADS, 1, 1);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = stream;
        // Programmatic dependent launch between the step's kernels: the launch latency of kernel N+1 overlaps kernel N
        // (measured on c2 against launches without it: gap A->B 2.9 -> 1.8 us, B->A 2.3 -> 1.95 us, step 22.25 -> 21.77 us).
        cudaLaunchAttribute at[2];
        at[0].id = cudaLaunchAttributePriority;
        at[0].val.priority = sn_high_priority();
        at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 2;
        RCN_LAUNCH(name, stream, cudaLaunchKernelEx(&cfg, kern, d, params, feats, Bi, onehot, labels, acts, deltas, stats_partial,
                                                    backward, front));
        return RCN_OK;
    };
    if (fr && fr->use_cp && fr->prewait && backward) {
        static SmemAttrCache attr;
        RCN_TRY(launch(smallnet_fwd_bwd_kernel<2, true>, attr,
                       fr->prewait == 2 ? "smallnet_fwd_bwd_kernel(fused features, front end ahead of the wait)"
                                        : "smallnet_fwd_bwd_kernel(fused features, front end ahead of the exchange)", *fr));
    } else if (fr && fr->use_cp) {
        static SmemAttrCache attr;
        RCN_TRY(launch(smallnet_fwd_bwd_kernel<2, false>, attr, "smallnet_fwd_bwd_kernel(fused features)", *fr));
    } else if (fr) {
        static SmemAttrCache attr;
        RCN_TRY(launch(smallnet_fwd_bwd_kernel<1, false>, attr, "smallnet_fwd_bwd_kernel(fused features)", *fr));
    } else {
        static SmemAttrCache attr;
        RCN_TRY(launch(smallnet_fwd_bwd_kernel<0, false>, attr, "smallnet_fwd_bwd_kernel", empty_front));
    }
    return RCN_OK;
}

int launch_smallnet_forward(const SmallNetDesc& d, const double* params, double* feats, size_t B, double* acts,
                            const SmallNetFront* front, cudaStream_t stream) {
    if (B == 0) return RCN_OK;
    return launch_kernel_a(d, params, feats, B, nullptr, nullptr, acts, nullptr, nullptr, 0, front, stream);
}

int launch_smallnet_infer(const SmallNetDesc& d, const double* params, size_t B, const int64_t* labels, int64_t* labels_out,
                          double* stats, ReduceScratch& ws, const SmallNetFront& front, cudaStream_t stream) {
    if (B == 0) return RCN_OK;
    const size_t chunk_max = smallnet_max_batch();
    RCN_TRY(ws.ensure(2 * (size_t)cdiv(B < chunk_max ? B : chunk_max, SN_TB) * sizeof(double), stream));
    SmallNetDesc di = d;
    di.tl = nullptr;                     // the launch timeline records the training kernels only
    const size_t smem = kernel_a_smem(d, &front);
    for (size_t c0 = 0; c0 < B; c0 += chunk_max) {
        const size_t n = B - c0 < chunk_max ? B - c0 : chunk_max;
        SnInfer inf{labels_out ? labels_out + c0 : nullptr, ws.tickets(), stats, c0 > 0 ? 1 : 0};
        SmallNetFront fr = front;
        fr.images += c0 * (size_t)fr.H * fr.W;
        auto launch = [&](auto kern, SmemAttrCache& attr, const char* name) -> int {
            if (attr.need(smem)) RCN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(cdiv(n, SN_TB), 1, 1);
            cfg.blockDim = dim3(SNA_THREADS, 1, 1);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = stream;
            // as the forward-only launch of kernel A: griddepcontrol.wait before any memory access, no early trigger
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            RCN_LAUNCH(name, stream, cudaLaunchKernelEx(&cfg, kern, di, params, (int)n, labels + c0, ws.partials(), inf, fr));
            return RCN_OK;
        };
        if (front.use_cp) {
            static SmemAttrCache attr;
            RCN_TRY(launch(smallnet_infer_kernel<2>, attr, "smallnet_infer_kernel(fused features)"));
        } else {
            static SmemAttrCache attr;
            RCN_TRY(launch(smallnet_infer_kernel<1>, attr, "smallnet_infer_kernel(fused features, generic front end)"));
        }
    }
    return RCN_OK;
}

int launch_smallnet_backprop(const SmallNetDesc& d, const double* params, double* feats, size_t B, const double* onehot,
                             const int64_t* labels, double* acts, double* deltas, double* grads, double* stats,
                             DevBuf& workspace, const SmallNetFront* front, cudaStream_t stream, const DpPush* dp_push,
                             const SnUpdate* update) {
    if (B == 0) return RCN_OK;
    if (B > smallnet_max_batch()) return fail(RCN_ERR_INVALID, "batch too large for the fused small-network path");
    int splits, ksplit;
    smallnet_splits(B, &splits, &ksplit);
    const int n_tiles = (int)cdiv(B, SN_TB);
    const int col_groups = (int)cdiv(d.n_in, 64);
    const int n_small = d.n_params - d.b_off[0];
    // workspace: per-tile statistics partials [n_tiles][2]
    RCN_TRY(workspace.reserve(2 * (size_t)n_tiles * sizeof(double)));
    double* stats_partial = workspace.as<double>();
    RCN_TRY(launch_kernel_a(d, params, feats, B, onehot, labels, acts, deltas, stats_partial, 1, front, stream));

    // dynamic smem of kernel B: the partial tile, and behind it the small CTA's staging area for `chunk` samples of the
    // narrow layers' activations and deltas (a whole K-split when it fits 96 KB: one pass, one L2 round trip)
    int per_sample = 0;
    for (int l = 0; l + 1 < d.n_layers; ++l) per_sample += d.rows[l];
    for (int l = 0; l < d.n_layers; ++l) per_sample += d.rows[l];
    int chunk = (int)((96 * 1024 / sizeof(double)) / (size_t)per_sample);
    if (chunk > ksplit) chunk = ksplit;
    if (chunk < 1) chunk = 1;
    const size_t tile_doubles = (size_t)(((n_small + 1) & ~1) > SNB_TILE ? ((n_small + 1) & ~1) : SNB_TILE);
    const size_t stg_doubles = (size_t)((n_small + 1) & ~1) + (size_t)chunk * per_sample;
    const size_t smem_b = (tile_doubles > stg_doubles ? tile_doubles : stg_doubles) * sizeof(double);
    DpPush push{};
    push.world = 1;
    if (dp_push) push = *dp_push;
    const bool with_push = push.world > 1;
    SnUpdate upd{};
    if (update) upd = *update;
    const int mode = with_push ? 1 : (upd.params ? 2 : 0);
    static SmemAttrCache attr_b;
    if (attr_b.need(smem_b)) {  // static 36 KB + dynamic tile exceeds the 48 KB default; all variants at once (a later
                                // launch of another variant may happen inside a stream capture)
        RCN_CUDA_TRY(cudaFuncSetAttribute(smallnet_wgrad_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        RCN_CUDA_TRY(cudaFuncSetAttribute(smallnet_wgrad_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        RCN_CUDA_TRY(cudaFuncSetAttribute(smallnet_wgrad_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    }
    cudaLaunchConfig_t cfg{};
    // one or two "small" column groups (db_l, dW_l of the narrow layers): two when there are more entries than threads and the
    // extra cluster still fits the single wave of ~15 eight-CTA clusters B200 co-schedules
    const int small_groups = (n_small > SNB_THREADS && (col_groups + 2) * splits <= 120) ? 2 : 1;
    cfg.gridDim = dim3(col_groups + small_groups, splits, 1);
    cfg.blockDim = dim3(SNB_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem_b;
    cfg.stream = stream;
    cudaLaunchAttribute attr[3];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = splits;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributePriority;
    attr[1].val.priority = sn_high_priority();
    attr[2].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[2].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 3;
    const int Bi = (int)B;
    auto kern = mode == 1 ? smallnet_wgrad_kernel<1> : mode == 2 ? smallnet_wgrad_kernel<2> : smallnet_wgrad_kernel<0>;
    RCN_LAUNCH(mode == 2 ? "smallnet_wgrad_kernel(+SGD update)" : "smallnet_wgrad_kernel", stream,
               cudaLaunchKernelEx(&cfg, kern, d, (const double*)feats, (const double*)acts, (const double*)deltas, Bi,
                                  ksplit, col_groups, grads, (const double*)stats_partial, n_tiles, stats, push, upd, chunk));
    return RCN_OK;
}

}  // namespace rcn

#ifdef RCN_SN_PHASES
extern "C" int rcn_cuda_debug_snp_stamps(long long* out /* [1024][8] */) {
    return cudaMemcpyFromSymbol(out, rcn::g_snp_stamp, sizeof(rcn::g_snp_stamp)) == cudaSuccess ? 0 : 4;
}
extern "C" int rcn_cuda_debug_sn_phases(long long* out /* [1024][32] */) {
    return cudaMemcpyFromSymbol(out, rcn::g_sn_phase, sizeof(rcn::g_sn_phase)) == cudaSuccess ? 0 : 4;
}
#endif
