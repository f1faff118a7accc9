// cnn.cuh -- what the convolutional network handle (cnn.cu) uses of the dense model it owns (model.cu).
#pragma once
#include "common.cuh"

namespace rcn {

// Forward pass of the dense stack on device features (cols[0] x B) as the model's evaluation runs it; then, where given,
// {the head's cost, hit count bits} of `labels` into stats[0..1] and the rcn.rs:92-97 argmax into labels_out (softmax head:
// of the logits, by softmax_xent_head_kernel).  Writes only
// the model's activations and scratch: gradients, deltas and the last-batch statistics stay as they are.
int model_evaluate_features(rcn_cuda_model* h, const double* feats, const int64_t* labels, size_t B, double* stats,
                            int64_t* labels_out);
// Output layer and cost of the model (RCN_HEAD_*): set before rcn_cuda_init_params_shapes, which then picks the route (the
// fused small-network kernels serve the sigmoid head only).  Not exported: the reference mirror RCN keeps rcn's head.
int model_set_head(rcn_cuda_model* h, int head);
// Device pointers of the first layer's weights W0 (rows0 x cols0, column-major) and of the first layer's deltas of the last
// accumulate (rows0 x B).
int model_first_layer(rcn_cuda_model* h, const double** W0, const double** delta0, size_t* rows0, size_t* cols0);
// Device pointer of the model's flat parameters [W0|b0|W1|b1|...] and their count: the optimizer step of the handle updates
// them in place (optim.cu).
int model_params(rcn_cuda_model* h, double** params, size_t* n);

}  // namespace rcn
