// smallnet.cuh -- fused training step for narrow sigmoid networks (every layer width <= 32), see smallnet.cu.
#pragma once
#include "common.cuh"
#include "features.cuh"
#include "timeline.cuh"

namespace rcn {

struct DpPush;   // dp.cuh: peers' receive slots, when the weight-gradient kernel pushes the exchange itself

constexpr int kSmallNetMaxLayers = 4;

struct SmallNetDesc {
    int n_layers;
    int n_in;                          // input width of layer 0 (feature length)
    int rows[kSmallNetMaxLayers];      // layer widths
    int w_off[kSmallNetMaxLayers];     // offsets into the flat [W0|b0|W1|b1|...] buffer
    int b_off[kSmallNetMaxLayers];
    int n_params;
    Timeline* tl;                      // device-side launch timeline (timeline.cuh), null = off
};

// Optional fused front end of kernel A: u8 images -> convpool stack -> standardised features, in shared memory.
struct SmallNetFront {
    const uint8_t* images;
    int H, W;
    int max_elems;                     // largest per-image map set any stage reads (elements)
    StageList stages;
    Standardise sc;
    BatchIndex bi;
    int prewait;                       // run the front end ahead of griddepcontrol.wait (smallnet.cu; needs use_cp).  1: data-parallel
                                       // step behind the exchange kernel (needs a cursor the previous kernel B advanced);
                                       // 2: one GPU, under the tail of the previous step's kernel B, which still reads the
                                       // feature buffer -- the features stay in the tile until the wait has passed
    int use_cp;                        // staged front end (bulk-async image loads, zero-framed tiles): see CpPlan
    int cp_pairs;                      // ... on image pairs in exact fp16 lanes (cp_item_pair): every intermediate is an integer of
                                       // magnitude <= 255 * 4^n_stages, which must not exceed 2048 -- one stage
    CpPlan cp;
};
// Fills use_cp / cp_pairs / cp: the staged front end needs a qualifying plan, 16-byte aligned images and H*W % 16 == 0.
void smallnet_front_select(const FeaturePlan& plan, SmallNetFront* fr);

// `params` may be null with `cursor` set: the kernel then only advances the cursor / writes the result ring (data-parallel
// groups, where the exchange kernel applies the update).
// Single-GPU steps fold the SGD update (rcn.rs:210-222) into the weight-gradient kernel: every CTA applies
// W -= scale * sum to exactly the elements whose batch sum it has just finished (one kernel and one launch gap less per
// step).  Also carries what sgd_update_kernel does on the side: the epoch cursor (rcn.rs:147) and the per-step result ring.
struct SnUpdate {
    double* params;          // nullptr = no fused update
    double scale;            // eta / B
    long long* cursor;       // optional epoch cursor, advanced by `batch` with chunks_exact wrap-around
    long long batch, n_samples;
    double* stats_ring;      // optional (pinned host) {cost, hits} per step
    int early_cursor;        // one GPU: advance the cursor BEFORE this kernel lets its dependents start (the next kernel A reads
                             // it ahead of its griddepcontrol.wait: SmallNetFront::prewait == 2)
};

bool smallnet_eligible(const SmallNetDesc& d);
size_t smallnet_max_batch();
bool smallnet_front_fits(const SmallNetDesc& d, const SmallNetFront& fr);

// acts: sum(rows) x B (layer after layer, rows_l x B column-major each), same layout for deltas.
// With a front end, `feats` (n_in x B) is an OUTPUT (kernel B and the parity taps read it); without, an input.
int launch_smallnet_forward(const SmallNetDesc& d, const double* params, double* feats, size_t B, double* acts,
                            const SmallNetFront* front, cudaStream_t stream);
// Test-set evaluation (rcn.rs:152-157) in the inference variant of kernel A, from the u8 images of `front`: stats[0..1] =
// quadratic cost and hit count (uint64 bits) of the whole batch, bit-identical to what launch_smallnet_backprop reports for
// it; labels_out (optional) the argmax of every sample.  The features never leave shared memory.  Batches above
// smallnet_max_batch() run as consecutive launches of that size.  Writes nothing else but `ws`.
int launch_smallnet_infer(const SmallNetDesc& d, const double* params, size_t B, const int64_t* labels, int64_t* labels_out,
                          double* stats, ReduceScratch& ws, const SmallNetFront& front, cudaStream_t stream);
// Full backprop of a minibatch: fills acts, deltas, the flat gradient buffer (batch sums) and stats[0..1]
// (quadratic cost, hit count as uint64 bits).
int launch_smallnet_backprop(const SmallNetDesc& d, const double* params, double* feats, size_t B, const double* onehot,
                             const int64_t* labels, double* acts, double* deltas, double* grads, double* stats,
                             DevBuf& workspace, const SmallNetFront* front, cudaStream_t stream,
                             const DpPush* dp_push = nullptr, const SnUpdate* update = nullptr);

}  // namespace rcn
