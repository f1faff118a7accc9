//! `extern "C"` bindings of include/rcn_cuda.h (1:1, hand-written; no bindgen needed).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_int, c_void};

#[repr(C)]
pub struct rcn_cuda_model {
    _private: [u8; 0],
}
pub type rcn_cuda_handle = *mut rcn_cuda_model;
#[repr(C)]
pub struct rcn_cuda_cnn {
    _private: [u8; 0],
}
pub type rcn_cuda_cnn_handle = *mut rcn_cuda_cnn;

pub const RCN_OK: c_int = 0;
pub const RCN_ERR_INVALID: c_int = 1;
pub const RCN_ERR_SHAPE: c_int = 2;
pub const RCN_ERR_NOT_IMPLEMENTED: c_int = 3;
pub const RCN_ERR_CUDA: c_int = 4;
pub const RCN_ERR_STATE: c_int = 5;
pub const RCN_ERR_OUT_OF_BOUNDS: c_int = 6;
pub const RCN_ERR_NAN: c_int = 7;
pub const RCN_PIXELS_U8_ROWMAJOR: c_int = 0;
pub const RCN_PIXELS_F64_COLMAJOR: c_int = 1;
pub const RCN_PIXELS_F64_NHWC: c_int = 2;
pub const RCN_CNN_CONV: i32 = 0;
pub const RCN_CNN_POOL: i32 = 1;
pub const RCN_CNN_LAYER_INTS: usize = 5;
pub const RCN_OPTIMIZER_SGD: c_int = 0;
pub const RCN_OPTIMIZER_ADAMW: c_int = 1;

extern "C" {
    pub fn rcn_cuda_last_error() -> *const c_char;
    pub fn rcn_cuda_create(classes: usize, convpool_cfg: *const i32, n_convpool: usize, feedforward_cfg: *const usize,
                           n_feedforward: usize, device: c_int, out: *mut rcn_cuda_handle) -> c_int;
    pub fn rcn_cuda_destroy(h: rcn_cuda_handle) -> c_int;
    pub fn rcn_cuda_feature_shape(h: rcn_cuda_handle, H: usize, W: usize, n_maps: *mut usize, map_h: *mut usize,
                                  map_w: *mut usize) -> c_int;
    pub fn rcn_cuda_init_params(h: rcn_cuda_handle, feature_len: usize) -> c_int;
    pub fn rcn_cuda_num_layers(h: rcn_cuda_handle, n: *mut usize) -> c_int;
    pub fn rcn_cuda_layer_shape(h: rcn_cuda_handle, layer: usize, rows: *mut usize, cols: *mut usize) -> c_int;
    pub fn rcn_cuda_set_weights(h: rcn_cuda_handle, layer: usize, rows: usize, cols: usize, w: *const c_double) -> c_int;
    pub fn rcn_cuda_get_weights(h: rcn_cuda_handle, layer: usize, w: *mut c_double) -> c_int;
    pub fn rcn_cuda_set_bias(h: rcn_cuda_handle, layer: usize, n: usize, b: *const c_double) -> c_int;
    pub fn rcn_cuda_get_bias(h: rcn_cuda_handle, layer: usize, b: *mut c_double) -> c_int;
    pub fn rcn_cuda_set_scale(h: rcn_cuda_handle, mean: c_double, sd: c_double) -> c_int;
    pub fn rcn_cuda_get_scale(h: rcn_cuda_handle, mean: *mut c_double, sd: *mut c_double) -> c_int;
    pub fn rcn_cuda_features(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, B: usize, H: usize, W: usize,
                             standardise: c_int, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_gen_scales(h: rcn_cuda_handle, feats: *const c_double, L: usize, B: usize, mean: *mut c_double,
                               sd: *mut c_double) -> c_int;
    pub fn rcn_cuda_standardise(h: rcn_cuda_handle, feats: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_forward(h: rcn_cuda_handle, feats: *const c_double, B: usize, out_acts: *mut c_double) -> c_int;
    pub fn rcn_cuda_classify(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, B: usize, H: usize, W: usize,
                             labels_out: *mut i64) -> c_int;
    pub fn rcn_cuda_evaluate(h: rcn_cuda_handle, feats: *const c_double, labels: *const i64, B: usize,
                             accept: *mut u64) -> c_int;
    pub fn rcn_cuda_evaluate_images(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                    B: usize, H: usize, W: usize, cost_out: *mut c_double, accept_out: *mut u64,
                                    labels_out: *mut i64) -> c_int;
    pub fn rcn_cuda_train_batch(h: rcn_cuda_handle, feats: *const c_double, onehot: *const c_double, labels: *const i64,
                                B: usize, eta: c_double) -> c_int;
    pub fn rcn_cuda_train_batch_images(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                       B: usize, H: usize, W: usize, eta: c_double) -> c_int;
    // ---- epoch loop over a host dataset, data-parallel group, checkpoint shapes -----------------------------------
    pub fn rcn_cuda_train_epoch_host(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                     n_samples: usize, H: usize, W: usize, B: usize, eta: c_double, global_batch: usize,
                                     cost_out: *mut c_double, hits_out: *mut u64, n_steps_out: *mut usize) -> c_int;
    pub fn rcn_cuda_dp_init(h: rcn_cuda_handle, world: c_int, rank: c_int, ipc_handle_out: *mut c_void) -> c_int;
    pub fn rcn_cuda_dp_connect_ipc(h: rcn_cuda_handle, all_handles: *const c_void) -> c_int;
    pub fn rcn_cuda_dp_connect_local(h: rcn_cuda_handle, group: *const rcn_cuda_handle) -> c_int;
    pub fn rcn_cuda_dp_shutdown(h: rcn_cuda_handle) -> c_int;
    pub fn rcn_cuda_dp_error(h: rcn_cuda_handle, error: *mut c_int) -> c_int;
    pub fn rcn_cuda_timeline_enable(h: rcn_cuda_handle, on: c_int) -> c_int;
    pub fn rcn_cuda_timeline_read(h: rcn_cuda_handle, stamps: *mut u64, launches: *mut u32) -> c_int;
    pub fn rcn_cuda_init_params_shapes(h: rcn_cuda_handle, rows: *const usize, cols: *const usize, n_layers: usize) -> c_int;
    pub fn rcn_cuda_accumulate_gradients_images(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int,
                                                labels: *const i64, B: usize, H: usize, W: usize) -> c_int;
    pub fn rcn_cuda_apply_gradients(h: rcn_cuda_handle, eta: c_double, batch: usize) -> c_int;
    pub fn rcn_cuda_last_batch_stats(h: rcn_cuda_handle, cost: *mut c_double, hits: *mut u64) -> c_int;
    // ---- extensions (not in the reference): learned conv, NHWC pooling, softmax cross-entropy, GEMM block ----------
    pub fn rcn_cuda_ext_conv2d_forward(device: c_int, stream: *mut c_void, x: *const c_double, B: usize, H: usize, W: usize,
                                       Ci: usize, w: *const c_double, bias: *const c_double, Co: usize, kh: usize, kw: usize,
                                       padding: c_int, activation: c_int, y: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_activation_backward(device: c_int, stream: *mut c_void, y: *const c_double, dy: *const c_double,
                                            n: usize, activation: c_int, dz: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_conv2d_backward_data(device: c_int, stream: *mut c_void, dz: *const c_double, B: usize, H: usize,
                                             W: usize, Ci: usize, w: *const c_double, Co: usize, kh: usize, kw: usize,
                                             padding: c_int, y_prev: *const c_double, activation_prev: c_int,
                                             dx: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_conv2d_backward_weight(device: c_int, stream: *mut c_void, x: *const c_double, dz: *const c_double,
                                               B: usize, H: usize, W: usize, Ci: usize, Co: usize, kh: usize, kw: usize,
                                               padding: c_int, dw: *mut c_double, db: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_pool2d_forward(device: c_int, stream: *mut c_void, x: *const c_double, B: usize, H: usize, W: usize,
                                       C: usize, padding: c_int, pooling: c_int, y: *mut c_double, argmax_out: *mut u8) -> c_int;
    pub fn rcn_cuda_ext_pool2d_backward(device: c_int, stream: *mut c_void, dy: *const c_double, argmax: *const u8, B: usize,
                                        H: usize, W: usize, C: usize, padding: c_int, pooling: c_int, dx: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_softmax_xent(device: c_int, stream: *mut c_void, z: *const c_double, n: usize, B: usize,
                                     onehot: *const c_double, labels: *const i64, probs: *mut c_double, loss: *mut c_double,
                                     delta: *mut c_double) -> c_int;
    pub fn rcn_cuda_ext_gemm_f64(device: c_int, stream: *mut c_void, A: *const c_double, lda: usize, a_kcontig: c_int,
                                 B: *const c_double, ldb: usize, b_kcontig: c_int, M: usize, N: usize, K: usize, impl_: c_int,
                                 C: *mut c_double) -> c_int;
    // ---- library / stream ------------------------------------------------------------------------------------------
    pub fn rcn_cuda_version() -> c_int;
    pub fn rcn_cuda_device_count(count: *mut c_int) -> c_int;
    pub fn rcn_cuda_set_stream(h: rcn_cuda_handle, cuda_stream: *mut c_void) -> c_int;
    pub fn rcn_cuda_synchronize(h: rcn_cuda_handle) -> c_int;
    // ---- flat parameter / gradient views (serialization.rs:19-22 order) ------------------------------------------------
    pub fn rcn_cuda_param_count(h: rcn_cuda_handle, n: *mut usize) -> c_int;
    pub fn rcn_cuda_set_params(h: rcn_cuda_handle, flat: *const c_double, n: usize) -> c_int;
    pub fn rcn_cuda_get_params(h: rcn_cuda_handle, flat: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_bind_gradient_buffer(h: rcn_cuda_handle, device_ptr: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_gradient_buffer(h: rcn_cuda_handle, device_ptr: *mut *mut c_double, n: *mut usize) -> c_int;
    pub fn rcn_cuda_get_gradients(h: rcn_cuda_handle, flat: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_get_activations(h: rcn_cuda_handle, layer: usize, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_get_deltas(h: rcn_cuda_handle, layer: usize, out: *mut c_double) -> c_int;
    // ---- classify_test argmax / backprop sums on features (rcn.rs:92-97, 190-205) --------------------------------------
    pub fn rcn_cuda_classify_features(h: rcn_cuda_handle, feats: *const c_double, B: usize, labels_out: *mut i64) -> c_int;
    pub fn rcn_cuda_accumulate_gradients(h: rcn_cuda_handle, feats: *const c_double, onehot: *const c_double,
                                         labels: *const i64, B: usize) -> c_int;
    // ---- epoch mode: chunks_exact loop over a dataset resident in HBM (rcn.rs:144-149) --------------------------------
    pub fn rcn_cuda_epoch_bind(h: rcn_cuda_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                               perm: *const i64, n_samples: usize, H: usize, W: usize, B: usize) -> c_int;
    pub fn rcn_cuda_epoch_seek(h: rcn_cuda_handle, position: usize) -> c_int;
    pub fn rcn_cuda_epoch_position(h: rcn_cuda_handle, position: *mut usize) -> c_int;
    pub fn rcn_cuda_epoch_accumulate(h: rcn_cuda_handle) -> c_int;
    pub fn rcn_cuda_epoch_apply(h: rcn_cuda_handle, eta: c_double, global_batch: usize) -> c_int;
    pub fn rcn_cuda_epoch_step(h: rcn_cuda_handle, eta: c_double) -> c_int;
    pub fn rcn_cuda_epoch_run(h: rcn_cuda_handle, eta: c_double, n_steps: usize) -> c_int;
    // ---- accounting ----------------------------------------------------------------------------------------------------
    pub fn rcn_cuda_kernel_launches(count: *mut u64) -> c_int;
    pub fn rcn_cuda_allocation_generation(generation: *mut u64) -> c_int;
    pub fn rcn_cuda_profile_enable(on: c_int) -> c_int;
    pub fn rcn_cuda_profile_report(json_out: *mut c_char, capacity: usize) -> c_int;
    // ---- op-level API: traits Convolve2D / Pool2D (kernel.rs:61-100, 219-236) ------------------------------------------
    pub fn rcn_cuda_convolve_2d(device: c_int, stream: *mut c_void, m: *const c_double, H: usize, W: usize,
                                kernel: *const c_double, kh: usize, kw: usize, padding: c_int, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_convolve_2d_separated(device: c_int, stream: *mut c_void, m: *const c_double, H: usize, W: usize,
                                          op: c_int, padding: c_int, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_relu(device: c_int, stream: *mut c_void, m: *const c_double, n: usize, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_pool_2d(device: c_int, stream: *mut c_void, m: *const c_double, H: usize, W: usize, padding: c_int,
                            pooling: c_int, out: *mut c_double, argmax_out: *mut u8) -> c_int;
    // ---- convolutional network handle (learned conv / pool layers + the dense stack) -------------------------------
    pub fn rcn_cuda_cnn_create(device: c_int, H: usize, W: usize, in_channels: usize, layer_spec: *const i32, n_layers: usize,
                               feedforward: *const usize, n_ff: usize, classes: usize, out: *mut rcn_cuda_cnn_handle) -> c_int;
    pub fn rcn_cuda_cnn_create_with_head(device: c_int, H: usize, W: usize, in_channels: usize, layer_spec: *const i32,
                                         n_layers: usize, feedforward: *const usize, n_ff: usize, classes: usize, head: c_int,
                                         out: *mut rcn_cuda_cnn_handle) -> c_int;
    pub fn rcn_cuda_cnn_destroy(h: rcn_cuda_cnn_handle) -> c_int;
    pub fn rcn_cuda_cnn_set_stream(h: rcn_cuda_cnn_handle, stream: *mut c_void) -> c_int;
    pub fn rcn_cuda_cnn_synchronize(h: rcn_cuda_cnn_handle) -> c_int;
    pub fn rcn_cuda_cnn_layer_shape(h: rcn_cuda_cnn_handle, layer: usize, H: *mut usize, W: *mut usize, C: *mut usize) -> c_int;
    pub fn rcn_cuda_cnn_param_count(h: rcn_cuda_cnn_handle, n: *mut usize) -> c_int;
    pub fn rcn_cuda_cnn_set_params(h: rcn_cuda_cnn_handle, flat: *const c_double, n: usize) -> c_int;
    pub fn rcn_cuda_cnn_get_params(h: rcn_cuda_cnn_handle, flat: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_cnn_accumulate(h: rcn_cuda_cnn_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                   B: usize, H: usize, W: usize) -> c_int;
    pub fn rcn_cuda_cnn_apply(h: rcn_cuda_cnn_handle, eta: c_double, global_batch: usize) -> c_int;
    pub fn rcn_cuda_cnn_train_batch(h: rcn_cuda_cnn_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                    B: usize, H: usize, W: usize, eta: c_double) -> c_int;
    pub fn rcn_cuda_cnn_last_batch_stats(h: rcn_cuda_cnn_handle, cost: *mut c_double, hits: *mut u64) -> c_int;
    pub fn rcn_cuda_cnn_epoch_bind(h: rcn_cuda_cnn_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                   perm: *const i64, n_samples: usize, H: usize, W: usize, B: usize) -> c_int;
    pub fn rcn_cuda_cnn_epoch_seek(h: rcn_cuda_cnn_handle, position: usize) -> c_int;
    pub fn rcn_cuda_cnn_epoch_position(h: rcn_cuda_cnn_handle, position: *mut usize) -> c_int;
    pub fn rcn_cuda_cnn_epoch_accumulate(h: rcn_cuda_cnn_handle) -> c_int;
    pub fn rcn_cuda_cnn_epoch_apply(h: rcn_cuda_cnn_handle, eta: c_double, global_batch: usize) -> c_int;
    pub fn rcn_cuda_cnn_epoch_step(h: rcn_cuda_cnn_handle, eta: c_double) -> c_int;
    pub fn rcn_cuda_cnn_epoch_run(h: rcn_cuda_cnn_handle, eta: c_double, n_steps: usize) -> c_int;
    pub fn rcn_cuda_cnn_evaluate_images(h: rcn_cuda_cnn_handle, images: *const c_void, pixel_format: c_int, labels: *const i64,
                                        B: usize, H: usize, W: usize, cost_out: *mut c_double, accept_out: *mut u64,
                                        labels_out: *mut i64) -> c_int;
    pub fn rcn_cuda_cnn_classify_images(h: rcn_cuda_cnn_handle, images: *const c_void, pixel_format: c_int, B: usize, H: usize,
                                        W: usize, labels_out: *mut i64) -> c_int;
    pub fn rcn_cuda_cnn_bind_gradient_buffer(h: rcn_cuda_cnn_handle, device_ptr: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_cnn_gradient_buffer(h: rcn_cuda_cnn_handle, device_ptr: *mut *mut c_double, n: *mut usize) -> c_int;
    pub fn rcn_cuda_cnn_get_gradients(h: rcn_cuda_cnn_handle, flat: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_cnn_get_layer_output(h: rcn_cuda_cnn_handle, layer: usize, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_cnn_get_input_gradient(h: rcn_cuda_cnn_handle, out: *mut c_double) -> c_int;
    pub fn rcn_cuda_cnn_set_optimizer(h: rcn_cuda_cnn_handle, kind: c_int, momentum: c_double, nesterov: c_int,
                                      weight_decay: c_double, beta1: c_double, beta2: c_double, eps: c_double) -> c_int;
    pub fn rcn_cuda_cnn_optimizer_state_size(h: rcn_cuda_cnn_handle, n: *mut usize) -> c_int;
    pub fn rcn_cuda_cnn_get_optimizer_state(h: rcn_cuda_cnn_handle, state: *mut c_double, n: usize) -> c_int;
    pub fn rcn_cuda_cnn_set_optimizer_state(h: rcn_cuda_cnn_handle, state: *const c_double, n: usize) -> c_int;
}
