//! Drop-in facade: the public API of `rcn` (rcn/src/rcn.rs, rcn/src/utils/kernel.rs) with the compute in
//! librcn_cuda.so. Same type names, argument meaning and panic behaviour as the CPU crate, so
//! `use rcn_cuda::{rcn::RCN, utils::kernel::*}` replaces `use rcn::{...}` in main.rs / benches / backend.
//! NOT compiled in this repository's environment (no rustc / cargo in the image): written against the crate versions of
//! rcn/Cargo.toml and kept in step with include/rcn_cuda.h by tests/test_abi.py::test_rust_extern_block_covers_header.
pub mod cuda;
pub mod ffi;
pub mod trainer;

use nalgebra::{DMatrix, DVector};
use std::ffi::CStr;
use std::ptr;

fn check(rc: i32) {
    if rc != ffi::RCN_OK {
        // contract violations panic exactly like the CPU crate (kernel.rs:127,133,200,247,284)
        let msg = unsafe { CStr::from_ptr(ffi::rcn_cuda_last_error()) }.to_string_lossy().into_owned();
        panic!("{msg}");
    }
}

pub mod utils {
    pub mod kernel {
        use super::super::{check, ffi};
        use nalgebra::DMatrix;
        use std::ptr;

        use serde::{Deserialize, Serialize};

        #[derive(Clone, Copy)]
        pub enum SeparableOperator { Top, Bottom, Left, Right }      // kernel.rs:16-21
        #[derive(Clone, Copy, Serialize, Deserialize)]
        pub enum Padding { None, Same }                              // kernel.rs:25-28 (variant index = bincode tag)
        #[derive(Clone, Copy, Serialize, Deserialize)]
        pub enum Pooling { Average, Max }                            // kernel.rs:32-35

        /// kernel.rs:61-100 -- implemented for DMatrix<f64> (the type the model uses).
        pub trait Convolve2D {
            fn convolve_2d(&self, kernel: &DMatrix<f64>, padding: &Padding) -> DMatrix<f64>;
            fn convolve_2d_separated(&self, op: SeparableOperator, padding: &Padding) -> DMatrix<f64>;
            fn relu(&self) -> DMatrix<f64>;
        }
        /// kernel.rs:219-236
        pub trait Pool2D {
            fn pool_2d(&self, padding: &Padding, pooling: &Pooling) -> DMatrix<f64>;
        }

        impl Convolve2D for DMatrix<f64> {
            fn convolve_2d(&self, kernel: &DMatrix<f64>, padding: &Padding) -> DMatrix<f64> {
                let (h, w) = self.shape();
                let (kh, kw) = kernel.shape();
                let (oh, ow) = match padding { Padding::Same => (h, w), Padding::None => (h + 1 - kh.min(h + 1), w + 1 - kw.min(w + 1)) };
                let mut out = DMatrix::<f64>::zeros(oh, ow);
                check(unsafe { ffi::rcn_cuda_convolve_2d(0, ptr::null_mut(), self.as_ptr(), h, w, kernel.as_ptr(), kh, kw,
                                                         *padding as i32, out.as_mut_ptr()) });
                out
            }
            fn convolve_2d_separated(&self, op: SeparableOperator, padding: &Padding) -> DMatrix<f64> {
                let (h, w) = self.shape();
                let (oh, ow) = match padding { Padding::Same => (h, w), Padding::None => (h.saturating_sub(2), w.saturating_sub(2)) };
                let mut out = DMatrix::<f64>::zeros(oh, ow);
                check(unsafe { ffi::rcn_cuda_convolve_2d_separated(0, ptr::null_mut(), self.as_ptr(), h, w, op as i32,
                                                                   *padding as i32, out.as_mut_ptr()) });
                out
            }
            fn relu(&self) -> DMatrix<f64> {
                let mut out = DMatrix::<f64>::zeros(self.nrows(), self.ncols());
                check(unsafe { ffi::rcn_cuda_relu(0, ptr::null_mut(), self.as_ptr(), self.len(), out.as_mut_ptr()) });
                out
            }
        }
        impl Pool2D for DMatrix<f64> {
            fn pool_2d(&self, padding: &Padding, pooling: &Pooling) -> DMatrix<f64> {
                let (h, w) = self.shape();
                let (oh, ow) = match padding { Padding::Same => ((h + 1) / 2, (w + 1) / 2), Padding::None => (h / 2, w / 2) };
                let mut out = DMatrix::<f64>::zeros(oh, ow);
                check(unsafe { ffi::rcn_cuda_pool_2d(0, ptr::null_mut(), self.as_ptr(), h, w, *padding as i32, *pooling as i32,
                                                     out.as_mut_ptr(), ptr::null_mut()) });
                out
            }
        }
    }
}

pub mod rcn {
    //! `RCN` with the reference's public surface (rcn.rs:58-64, 82, 126-133) and its bincode byte layout. The parameters
    //! live in HBM behind the handle; `layer_weights` / `layer_bias` / `scale_set` exist on the host only while a model
    //! is being (de)serialised.
    use super::cuda::{DeviceBuffer, PinnedBuffer};
    use super::utils::kernel::{Padding, Pooling};
    use super::{check, ffi, DMatrix, DVector};
    use image::{io::Reader as ImageReader, DynamicImage, ImageError};
    use rand::{seq::SliceRandom, Rng};
    use rand_distr::StandardNormal;
    use serde::{de::Deserializer, ser::Serializer, Deserialize, Serialize};
    use std::os::raw::c_void;
    use std::sync::Mutex;
    use std::path::{Path, PathBuf};
    use std::{fs, ptr};

    /// rcn.rs:35-38
    #[derive(Clone, Copy, Serialize, Deserialize)]
    pub enum RCNLayer { Convolve2D(Padding), Pool2D(Pooling) }
    /// rcn.rs:28-31
    pub struct Weights(pub DMatrix<f64>);
    pub struct Bias(pub DVector<f64>);

    // serialization.rs:11-24,98: struct { dims: (usize, usize), data: Vec<f64> (column-major) }
    #[derive(Serialize, Deserialize)]
    #[serde(rename = "Weights")]
    struct WeightsRepr { dims: (usize, usize), data: Vec<f64> }
    impl Serialize for Weights {
        fn serialize<S: Serializer>(&self, s: S) -> Result<S::Ok, S::Error> {
            WeightsRepr { dims: self.0.shape(), data: self.0.as_slice().to_vec() }.serialize(s)
        }
    }
    impl<'de> Deserialize<'de> for Weights {
        fn deserialize<D: Deserializer<'de>>(d: D) -> Result<Self, D::Error> {
            let r = WeightsRepr::deserialize(d)?;
            if r.data.len() != r.dims.0 * r.dims.1 {
                return Err(serde::de::Error::custom("Weights: data length does not match dims"));
            }
            Ok(Weights(DMatrix::from_vec(r.dims.0, r.dims.1, r.data)))
        }
    }
    // serialization.rs:104-151: a plain sequence of f64
    impl Serialize for Bias {
        fn serialize<S: Serializer>(&self, s: S) -> Result<S::Ok, S::Error> { self.0.as_slice().serialize(s) }
    }
    impl<'de> Deserialize<'de> for Bias {
        fn deserialize<D: Deserializer<'de>>(d: D) -> Result<Self, D::Error> {
            Ok(Bias(DVector::from_vec(Vec::<f64>::deserialize(d)?)))
        }
    }

    /// The reference's struct, field for field (rcn.rs:13-25): what `rcn.bin` holds.
    #[derive(Serialize, Deserialize)]
    #[serde(rename = "RCN")]
    struct Checkpoint<'a> {
        classes: usize,
        convpool_cfg: Vec<RCNLayer>,
        feedforward_cfg: Vec<usize>,
        layer_weights: Vec<Weights>,
        layer_bias: Vec<Bias>,
        scale_set: (f64, f64),
        training_path: &'a str,
        testing_path: &'a str,
    }

    /// One decoded data set on the host: N images of h x w Luma8 bytes, row-major, in page-locked memory.
    struct HostSet { pixels: PinnedBuffer<u8>, labels: Vec<i64>, n: usize, h: usize, w: usize }

    pub struct RCN<'a> {
        handle: ffi::rcn_cuda_handle,
        device: i32,
        classes: usize,
        convpool_cfg: Vec<RCNLayer>,
        feedforward_cfg: Vec<usize>,
        training_path: &'a str,
        testing_path: &'a str,
        // `&self` entry points (classify) use the handle's scratch buffers: one caller at a time, like the mutexes the
        // reference takes inside train_batch (rcn.rs:185-186). Mutation goes through `&mut self`.
        gate: Mutex<()>,
    }

    fn layer_code(l: &RCNLayer) -> i32 {
        match l {
            RCNLayer::Convolve2D(p) => *p as i32,          // RCN_LAYER_CONV_NONE / _SAME
            RCNLayer::Pool2D(p) => 2 + *p as i32,          // RCN_LAYER_POOL_AVERAGE / _MAX
        }
    }

    /// `get_pixel_matrix` (lib.rs:27-41) without the f64 detour: Luma8 / LumaA8 -> h*w bytes, anything else is the
    /// reference's InvalidGrayscaleImageError (which `load_data` unwraps into a panic, rcn.rs:400).
    fn luma_bytes(img: DynamicImage) -> Result<(Vec<u8>, usize, usize), &'static str> {
        match img {
            DynamicImage::ImageLuma8(g) => { let (w, h) = g.dimensions(); Ok((g.into_raw(), h as usize, w as usize)) }
            DynamicImage::ImageLumaA8(g) => {
                let (w, h) = g.dimensions();
                Ok((g.into_raw().chunks_exact(2).map(|p| p[0]).collect(), h as usize, w as usize))
            }
            _ => Err("InvalidGrayscaleImageError: Image provided was not Luma8 (grayscaled image)"),
        }
    }

    impl<'a> RCN<'a> {
        /// rcn.rs:58-64
        pub fn new(classes: usize, convpool_cfg: Vec<RCNLayer>, feedforward_cfg: Vec<usize>, training_path: &'a str,
                   testing_path: &'a str) -> Self {
            Self::on_device(0, classes, convpool_cfg, feedforward_cfg, training_path, testing_path)
        }

        /// Same model on GPU `device` (one replica per GPU for the data-parallel trainer).
        pub fn on_device(device: i32, classes: usize, convpool_cfg: Vec<RCNLayer>, feedforward_cfg: Vec<usize>,
                         training_path: &'a str, testing_path: &'a str) -> Self {
            let codes: Vec<i32> = convpool_cfg.iter().map(layer_code).collect();
            let mut handle = ptr::null_mut();
            check(unsafe { ffi::rcn_cuda_create(classes, codes.as_ptr(), codes.len(), feedforward_cfg.as_ptr(),
                                                feedforward_cfg.len(), device, &mut handle) });
            RCN { handle, device, classes, convpool_cfg, feedforward_cfg, training_path, testing_path, gate: Mutex::new(()) }
        }

        pub(crate) fn raw(&self) -> ffi::rcn_cuda_handle { self.handle }
        pub fn device(&self) -> i32 { self.device }

        /// Number of dense layers; 0 while the model has no parameters yet (`layer_weights.is_empty()`, rcn.rs:139).
        fn num_layers(&self) -> usize {
            let mut n = 0usize;
            let rc = unsafe { ffi::rcn_cuda_num_layers(self.handle, &mut n) };
            if rc == ffi::RCN_ERR_STATE { return 0; }
            check(rc);
            n
        }

        pub fn scale_set(&self) -> (f64, f64) {
            let (mut m, mut s) = (0f64, 0f64);
            check(unsafe { ffi::rcn_cuda_get_scale(self.handle, &mut m, &mut s) });
            (m, s)
        }

        fn set_scale(&mut self, ms: (f64, f64)) { check(unsafe { ffi::rcn_cuda_set_scale(self.handle, ms.0, ms.1) }); }

        /// rcn.rs:82-98: decode on the host; features, standardise, forward and argmax (last max wins) on the GPU.
        pub fn classify(&self, img_path: &str) -> Result<usize, Box<dyn std::error::Error>> {
            let img = ImageReader::open(img_path)?.decode()?.grayscale();
            let (bytes, h, w) = luma_bytes(img).map_err(|e| Box::<dyn std::error::Error>::from(e))?;
            let mut label = 0i64;
            let _one_at_a_time = self.gate.lock().unwrap();
            check(unsafe { ffi::rcn_cuda_classify(self.handle, bytes.as_ptr() as *const c_void, ffi::RCN_PIXELS_U8_ROWMAJOR,
                                                  1, h, w, &mut label) });
            Ok(label as usize)
        }

        /// rcn.rs:152-157 on `n` decoded h x w Luma8 images (row-major, back to back) standardised with scale_set:
        /// (accept, quadratic cost sum_b 0.5*|a - y|^2) in one call, without materialising the features.
        pub fn evaluate_images(&self, pixels: &[u8], labels: &[i64], n: usize, h: usize, w: usize) -> (u64, f64) {
            assert!(pixels.len() == n * h * w && labels.len() == n, "evaluate_images: {} images of {}x{} expected", n, h, w);
            let (mut accept, mut cost) = (0u64, 0f64);
            let _one_at_a_time = self.gate.lock().unwrap();
            check(unsafe { ffi::rcn_cuda_evaluate_images(self.handle, pixels.as_ptr() as *const c_void,
                                                         ffi::RCN_PIXELS_U8_ROWMAJOR, labels.as_ptr(), n, h, w, &mut cost,
                                                         &mut accept, ptr::null_mut()) });
            (accept, cost)
        }

        /// rcn.rs:126-167. Host: directory walk, sampling, PNG decode, shuffle. GPU: everything else -- the feature
        /// stage and the statistics of each set, the `chunks_exact` loop (one call per epoch, the next chunk is pulled
        /// over PCIe while the current one trains) and the per-epoch evaluation on the HBM-resident test features.
        pub fn train(&mut self, batch_size: usize, epochs: usize, eta: f64, training_class_size_limit: usize,
                     testing_class_size_limit: usize) -> Result<(), ImageError> {
            let training = self.load_data(self.training_path, training_class_size_limit);
            let train_scale = self.scale_set();      // the training steps standardise with the training set's statistics
            let testing = self.load_data(self.testing_path, testing_class_size_limit);
            let test_scale = self.scale_set();       // ... and scale_set ends up holding the TEST set's (rcn.rs:134-137,406)

            let feature_len = self.feature_len(training.h, training.w);
            if self.num_layers() == 0 {
                self.load_weights_and_bias(feature_len);                                     // rcn.rs:139-141
            }

            // test features: computed once, standardised with the test statistics, resident in HBM for every epoch
            let mut test_feats = DeviceBuffer::<f64>::new(self.device, feature_len * testing.n);
            let test_labels = DeviceBuffer::<i64>::from_slice(self.device, &testing.labels);
            check(unsafe { ffi::rcn_cuda_features(self.handle, testing.pixels.as_ptr() as *const c_void,
                                                  ffi::RCN_PIXELS_U8_ROWMAJOR, testing.n, testing.h, testing.w, 1,
                                                  test_feats.as_mut_ptr()) });

            let img = training.h * training.w;
            let mut order: Vec<usize> = (0..training.n).collect();
            let mut shuffled = PinnedBuffer::<u8>::new(training.n * img);
            let mut shuffled_labels = vec![0i64; training.n];
            for e in 0..epochs {
                order.shuffle(&mut rand::thread_rng());                                      // rcn.rs:146
                for (dst, &src) in order.iter().enumerate() {
                    shuffled.as_mut_slice()[dst * img..(dst + 1) * img]
                        .copy_from_slice(&training.pixels.as_slice()[src * img..(src + 1) * img]);
                    shuffled_labels[dst] = training.labels[src];
                }
                self.set_scale(train_scale);
                let mut steps = 0usize;
                // for batch in training_set.chunks_exact(batch_size) { self.train_batch(batch, eta) }   (rcn.rs:147-149)
                check(unsafe { ffi::rcn_cuda_train_epoch_host(self.handle, shuffled.as_ptr() as *const c_void,
                                                              ffi::RCN_PIXELS_U8_ROWMAJOR, shuffled_labels.as_ptr(),
                                                              training.n, training.h, training.w, batch_size, eta, 0,
                                                              ptr::null_mut(), ptr::null_mut(), &mut steps) });
                self.set_scale(test_scale);
                let mut accept = 0u64;                                                       // rcn.rs:152-157
                check(unsafe { ffi::rcn_cuda_evaluate(self.handle, test_feats.as_ptr(), test_labels.as_ptr(), testing.n,
                                                      &mut accept) });
                println!("Epoch {}: {}/{} [{:.2}%]", e, accept, testing.n,
                         (accept as f64 / testing.n as f64) * 100_f64);                      // rcn.rs:158-164
            }
            Ok(())
        }

        fn feature_len(&self, h: usize, w: usize) -> usize {
            let (mut maps, mut mh, mut mw) = (0usize, 0usize, 0usize);
            check(unsafe { ffi::rcn_cuda_feature_shape(self.handle, h, w, &mut maps, &mut mh, &mut mw) });
            maps * mh * mw
        }

        /// rcn.rs:367-415: class directories in sorted order, `class_size_limit` files per class drawn uniformly without
        /// replacement, decoded to grayscale; then gen_scales over the raw features of the whole set (stored as scale_set).
        /// All pixels of the set land in ONE page-locked buffer so that the GPU can stream it.
        fn load_data(&mut self, path: &str, class_size_limit: usize) -> HostSet {
            fn entries(dir: &Path) -> Vec<PathBuf> {
                let mut v: Vec<PathBuf> = fs::read_dir(dir)
                    .unwrap_or_else(|e| panic!("cannot read {}: {e}", dir.display()))
                    .map(|entry| entry.expect("directory entry").path())
                    .collect();
                v.sort();
                v
            }
            let mut rng = rand::thread_rng();
            let mut staged: Vec<u8> = Vec::new();
            let mut labels: Vec<i64> = Vec::new();
            let mut dims: Option<(usize, usize)> = None;
            for (class_index, dir) in entries(Path::new(path)).iter().enumerate() {
                let mut files = entries(dir);
                if class_size_limit > files.len() {
                    // same message as the reference's panic (rcn.rs:383-390)
                    panic!("provided class_size_limit for {} too large! expected {} <= {}", path, class_size_limit, files.len());
                }
                let (chosen, _rest) = files.partial_shuffle(&mut rng, class_size_limit);
                for file in chosen.iter() {
                    let decoded = ImageReader::open(file).unwrap().decode().unwrap().grayscale();
                    let (px, ih, iw) = luma_bytes(decoded).unwrap();
                    let (h, w) = *dims.get_or_insert((ih, iw));
                    assert!(ih == h && iw == w, "all images of a data set must have the same size ({h}x{w}), got {ih}x{iw}");
                    staged.extend_from_slice(&px);
                    labels.push(class_index as i64);
                }
            }
            let (h, w) = dims.expect("empty data set");
            let n = labels.len();
            let mut pixels = PinnedBuffer::<u8>::new(staged.len());
            pixels.as_mut_slice().copy_from_slice(&staged);
            // gen_scales (rcn.rs:230-251) on the device: raw features of the whole set, then mean / population sd
            let l = self.feature_len(h, w);
            let mut feats = DeviceBuffer::<f64>::new(self.device, l * n);
            check(unsafe { ffi::rcn_cuda_features(self.handle, pixels.as_ptr() as *const c_void, ffi::RCN_PIXELS_U8_ROWMAJOR,
                                                  n, h, w, 0, feats.as_mut_ptr()) });
            let (mut mean, mut sd) = (0f64, 0f64);
            check(unsafe { ffi::rcn_cuda_gen_scales(self.handle, feats.as_ptr(), l, n, &mut mean, &mut sd) });
            HostSet { pixels, labels, n, h, w }
        }

        /// rcn.rs:425-457 + 500-523: the reference's shapes (including its `4^c / 2^p * l` first width, computed by the
        /// library) filled with unscaled N(0,1) draws, column-major.
        fn load_weights_and_bias(&mut self, l: usize) {
            check(unsafe { ffi::rcn_cuda_init_params(self.handle, l) });
            let mut rng = rand::thread_rng();
            for layer in 0..self.num_layers() {
                let (mut r, mut c) = (0usize, 0usize);
                check(unsafe { ffi::rcn_cuda_layer_shape(self.handle, layer, &mut r, &mut c) });
                let w: Vec<f64> = (0..r * c).map(|_| rng.sample(StandardNormal)).collect();
                let b: Vec<f64> = (0..r).map(|_| rng.sample(StandardNormal)).collect();
                check(unsafe { ffi::rcn_cuda_set_weights(self.handle, layer, r, c, w.as_ptr()) });
                check(unsafe { ffi::rcn_cuda_set_bias(self.handle, layer, r, b.as_ptr()) });
            }
        }

        /// Weights / Bias of one layer, read back from HBM (column-major: `DMatrix::from_vec` takes it as is).
        pub fn layer_weights(&self, layer: usize) -> Weights {
            let (mut r, mut c) = (0usize, 0usize);
            check(unsafe { ffi::rcn_cuda_layer_shape(self.handle, layer, &mut r, &mut c) });
            let mut m = DMatrix::<f64>::zeros(r, c);
            check(unsafe { ffi::rcn_cuda_get_weights(self.handle, layer, m.as_mut_ptr()) });
            Weights(m)
        }
        pub fn layer_bias(&self, layer: usize) -> Bias {
            let (mut r, mut c) = (0usize, 0usize);
            check(unsafe { ffi::rcn_cuda_layer_shape(self.handle, layer, &mut r, &mut c) });
            let mut v = DVector::<f64>::zeros(r);
            check(unsafe { ffi::rcn_cuda_get_bias(self.handle, layer, v.as_mut_ptr()) });
            Bias(v)
        }
    }

    /// `bincode::serialize(&model)` (main.rs:77): same bytes as the CPU crate writes.
    impl<'a> Serialize for RCN<'a> {
        fn serialize<S: Serializer>(&self, s: S) -> Result<S::Ok, S::Error> {
            let _one_at_a_time = self.gate.lock().unwrap();
            let n = self.num_layers();
            Checkpoint {
                classes: self.classes,
                convpool_cfg: self.convpool_cfg.clone(),
                feedforward_cfg: self.feedforward_cfg.clone(),
                layer_weights: (0..n).map(|l| self.layer_weights(l)).collect(),
                layer_bias: (0..n).map(|l| self.layer_bias(l)).collect(),
                scale_set: self.scale_set(),
                training_path: self.training_path,
                testing_path: self.testing_path,
            }.serialize(s)
        }
    }

    /// `bincode::deserialize(&data[..])` (main.rs:50, backend/src/main.rs:68): the file, not the config, decides the
    /// matrices; they go straight to HBM.
    impl<'de: 'a, 'a> Deserialize<'de> for RCN<'a> {
        fn deserialize<D: Deserializer<'de>>(d: D) -> Result<Self, D::Error> {
            let c = Checkpoint::deserialize(d)?;
            let mut m = RCN::new(c.classes, c.convpool_cfg, c.feedforward_cfg, c.training_path, c.testing_path);
            if !c.layer_weights.is_empty() {
                let rows: Vec<usize> = c.layer_weights.iter().map(|w| w.0.nrows()).collect();
                let cols: Vec<usize> = c.layer_weights.iter().map(|w| w.0.ncols()).collect();
                check(unsafe { ffi::rcn_cuda_init_params_shapes(m.handle, rows.as_ptr(), cols.as_ptr(), rows.len()) });
                for (l, (w, b)) in c.layer_weights.iter().zip(c.layer_bias.iter()).enumerate() {
                    check(unsafe { ffi::rcn_cuda_set_weights(m.handle, l, rows[l], cols[l], w.0.as_ptr()) });
                    check(unsafe { ffi::rcn_cuda_set_bias(m.handle, l, b.0.len(), b.0.as_ptr()) });
                }
            }
            m.set_scale(c.scale_set);
            Ok(m)
        }
    }

    impl<'a> Drop for RCN<'a> {
        fn drop(&mut self) { unsafe { ffi::rcn_cuda_destroy(self.handle); } }
    }
    // The handle is an owned heap object with no thread affinity (every entry point selects its device itself); `&self`
    // entry points serialise on `gate`, so the `Sync` the CPU crate relies on (rcn.rs:190-191, actix workers) holds.
    unsafe impl<'a> Send for RCN<'a> {}
    unsafe impl<'a> Sync for RCN<'a> {}
}
