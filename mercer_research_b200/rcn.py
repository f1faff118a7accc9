"""Host-side mirror of rcn's model layer (rcn/src/rcn.rs): ``RCN``, ``RCNLayer``, ``Weights`` / ``Bias`` access,
``train`` / ``classify`` -- same names, argument meaning and error behaviour -- driving librcn_cuda.so.

Batches are numpy arrays (staged through the device) or torch CUDA tensors (used in place, on torch's current
stream):  images ``(B, H, W)`` uint8 (the `image` crate's row-major Luma8 buffer) or float64 ``(B, H, W)`` indexed
(row, col); features ``(B, L)`` float64; labels ``(B,)`` int64; one-hot targets ``(B, classes)`` float64.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from .kernel import Padding, Pooling, _is_torch


@dataclass(frozen=True)
class RCNLayer:
    """``enum RCNLayer { Convolve2D(Padding), Pool2D(Pooling) }`` (rcn.rs:35-38)."""
    kind: str
    arg: int

    @staticmethod
    def Convolve2D(padding: Padding) -> "RCNLayer":
        return RCNLayer("Convolve2D", int(Padding(padding)))

    @staticmethod
    def Pool2D(pooling: Pooling) -> "RCNLayer":
        return RCNLayer("Pool2D", int(Pooling(pooling)))

    @property
    def code(self) -> int:
        """RCN_LAYER_* code of include/rcn_cuda.h."""
        return self.arg if self.kind == "Convolve2D" else 2 + self.arg


def _layer_code(layer) -> int:
    return layer.code if isinstance(layer, RCNLayer) else int(layer)


class _Buf:
    """Pointer + keep-alive for a host (numpy) or device (torch) buffer."""

    def __init__(self, x, dtype, shape_tail=None):
        if _is_torch(x):
            import torch
            tdt = {np.float64: torch.float64, np.uint8: torch.uint8, np.int64: torch.int64}[dtype]
            if not x.is_cuda:
                raise ValueError("torch tensors must live on a CUDA device (pass numpy arrays for host data)")
            self.store = x.to(tdt).contiguous()
            self.ptr = self.store.data_ptr()
            self.shape = tuple(self.store.shape)
            self.torch = True
            self.device = x.device
        else:
            self.store = np.ascontiguousarray(x, dtype=dtype)
            self.ptr = self.store.ctypes.data
            self.shape = self.store.shape
            self.torch = False
            self.device = None


class RCN:
    """Rust Convolutional Neural Network on a B200 (rcn.rs:15-25).

    ``training_path`` / ``testing_path`` are kept for API parity with ``RCN::new`` (rcn.rs:58-64); the array entry
    points below take data directly.
    """

    def __init__(self, classes: int, convpool_cfg: Sequence, feedforward_cfg: Sequence[int],
                 training_path: str = "", testing_path: str = "", device: int = 0):
        self._lib = _lib.load()
        self.classes = int(classes)
        self.convpool_cfg = list(convpool_cfg)
        self.feedforward_cfg = [int(x) for x in feedforward_cfg]
        self.training_path = training_path
        self.testing_path = testing_path
        self.device = int(device)
        codes = [_layer_code(l) for l in self.convpool_cfg]
        cfg = (C.c_int32 * max(1, len(codes)))(*codes)
        ff = (C.c_size_t * max(1, len(self.feedforward_cfg)))(*self.feedforward_cfg)
        h = C.c_void_p()
        _lib.check(self._lib.rcn_cuda_create(self.classes, cfg, len(codes), ff, len(self.feedforward_cfg), self.device,
                                             C.byref(h)))
        self._h = h
        self._shapes: List[Tuple[int, int]] = []

    # -- lifetime ---------------------------------------------------------------------------------------------
    def save(self, path: str = "./rcn.bin"):
        """``fs::write("./rcn.bin", bincode::serialize(&model)?)`` (main.rs:77), byte-compatible with the reference."""
        from . import serialization
        serialization.save(self, path)

    @staticmethod
    def load(path: str = "./rcn.bin", device: int = 0) -> "RCN":
        """``bincode::deserialize`` of a reference (or own) checkpoint onto a B200 (main.rs:47-50)."""
        from . import serialization
        return serialization.load(path, device=device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rcn_cuda_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: Optional[int]):
        """Run on an existing cudaStream_t (int handle, e.g. ``torch.cuda.current_stream().cuda_stream``; 0 / None is
        the CUDA legacy default stream). ``set_stream(-1)`` restores the model's private stream."""
        if cuda_stream is not None and cuda_stream < 0:
            cuda_stream = C.c_void_p(-1).value
        _lib.check(self._lib.rcn_cuda_set_stream(self._h, cuda_stream))

    def synchronize(self):
        _lib.check(self._lib.rcn_cuda_synchronize(self._h))

    def _use_torch_stream(self, *bufs):
        for b in bufs:
            if b is not None and b.torch:
                import torch
                self.set_stream(torch.cuda.current_stream(b.device).cuda_stream)
                return

    # -- shapes / parameters ----------------------------------------------------------------------------------
    def feature_shape(self, H: int, W: int) -> Tuple[int, int, int]:
        """(n_maps, map_h, map_w) of flatten_feature_set (rcn.rs:317-356) for an H x W image."""
        n, h, w = C.c_size_t(), C.c_size_t(), C.c_size_t()
        _lib.check(self._lib.rcn_cuda_feature_shape(self._h, H, W, C.byref(n), C.byref(h), C.byref(w)))
        return n.value, h.value, w.value

    def feature_len(self, H: int, W: int) -> int:
        n, h, w = self.feature_shape(H, W)
        return n * h * w

    def load_weights_and_bias(self, l: int):
        """rcn.rs:425-457: allocate the reference's layer shapes for feature length ``l`` (zero-filled; inject
        values with set_weights / set_bias / set_params)."""
        _lib.check(self._lib.rcn_cuda_init_params(self._h, int(l)))
        n = C.c_size_t()
        _lib.check(self._lib.rcn_cuda_num_layers(self._h, C.byref(n)))
        self._shapes = []
        for i in range(n.value):
            r, c = C.c_size_t(), C.c_size_t()
            _lib.check(self._lib.rcn_cuda_layer_shape(self._h, i, C.byref(r), C.byref(c)))
            self._shapes.append((r.value, c.value))

    def load_weights_and_bias_shapes(self, shapes):
        """Explicit (rows, cols) per layer, for a model restored from a checkpoint (serialization.py)."""
        rows = (C.c_size_t * len(shapes))(*[int(s[0]) for s in shapes])
        cols = (C.c_size_t * len(shapes))(*[int(s[1]) for s in shapes])
        _lib.check(self._lib.rcn_cuda_init_params_shapes(self._h, rows, cols, len(shapes)))
        self._shapes = [(int(s[0]), int(s[1])) for s in shapes]

    def _require_params(self):
        if not self._shapes:  # raises RCN_ERR_STATE from the library
            n = C.c_size_t()
            _lib.check(self._lib.rcn_cuda_param_count(self._h, C.byref(n)))

    @property
    def layer_shapes(self) -> List[Tuple[int, int]]:
        return list(self._shapes)

    @property
    def n_params(self) -> int:
        return sum(r * c + r for r, c in self._shapes)

    def set_weights(self, layer: int, w):
        """``Weights`` (rcn.rs:28): (rows, cols) matrix, stored column-major like nalgebra."""
        w = np.asarray(w, dtype=np.float64)
        buf = np.asfortranarray(w)
        _lib.check(self._lib.rcn_cuda_set_weights(self._h, layer, w.shape[0], w.shape[1], buf.ctypes.data))

    def get_weights(self, layer: int) -> np.ndarray:
        r, c = self._shapes[layer]
        buf = np.zeros((r, c), order="F")
        _lib.check(self._lib.rcn_cuda_get_weights(self._h, layer, buf.ctypes.data))
        return buf

    def set_bias(self, layer: int, b):
        b = np.ascontiguousarray(b, dtype=np.float64).ravel()
        _lib.check(self._lib.rcn_cuda_set_bias(self._h, layer, b.size, b.ctypes.data))

    def get_bias(self, layer: int) -> np.ndarray:
        buf = np.zeros(self._shapes[layer][0])
        _lib.check(self._lib.rcn_cuda_get_bias(self._h, layer, buf.ctypes.data))
        return buf

    def set_params(self, flat):
        flat = np.ascontiguousarray(flat, dtype=np.float64).ravel()
        _lib.check(self._lib.rcn_cuda_set_params(self._h, flat.ctypes.data, flat.size))

    def get_params(self) -> np.ndarray:
        self._require_params()
        buf = np.zeros(self.n_params)
        _lib.check(self._lib.rcn_cuda_get_params(self._h, buf.ctypes.data, buf.size))
        return buf

    def get_gradients(self) -> np.ndarray:
        self._require_params()
        buf = np.zeros(self.n_params)
        _lib.check(self._lib.rcn_cuda_get_gradients(self._h, buf.ctypes.data, buf.size))
        return buf

    @property
    def scale_set(self) -> Tuple[float, float]:
        m, s = C.c_double(), C.c_double()
        _lib.check(self._lib.rcn_cuda_get_scale(self._h, C.byref(m), C.byref(s)))
        return m.value, s.value

    @scale_set.setter
    def scale_set(self, ms):
        _lib.check(self._lib.rcn_cuda_set_scale(self._h, float(ms[0]), float(ms[1])))

    # -- feature stage ----------------------------------------------------------------------------------------
    def _images(self, images):
        if _is_torch(images):
            import torch
            if images.dtype == torch.uint8:
                b = _Buf(images, np.uint8)
                return b, _lib.PIXELS_U8_ROWMAJOR, b.shape
            b = _Buf(images.transpose(1, 2), np.float64)  # (B, W, H) contiguous == column-major H x W images
            return b, _lib.PIXELS_F64_COLMAJOR, (b.shape[0], b.shape[2], b.shape[1])
        a = np.asarray(images)
        if a.ndim != 3:
            raise ValueError("images must be (B, H, W)")
        if a.dtype == np.uint8:
            b = _Buf(a, np.uint8)
            return b, _lib.PIXELS_U8_ROWMAJOR, a.shape
        b = _Buf(np.ascontiguousarray(np.transpose(a, (0, 2, 1)), dtype=np.float64), np.float64)
        return b, _lib.PIXELS_F64_COLMAJOR, a.shape

    def flatten_feature_set(self, images, standardise: bool = False, out=None):
        """rcn.rs:317-356 over a batch (optionally followed by the standardise+clamp of rcn.rs:407-412 with
        ``scale_set``). Returns (B, L) float64 -- numpy for numpy input, a torch CUDA tensor for torch input."""
        buf, fmt, (B, H, W) = self._images(images)
        L = self.feature_len(H, W)
        self._use_torch_stream(buf)
        if buf.torch:
            import torch
            o = out if out is not None else torch.empty((B, L), dtype=torch.float64, device=buf.device)
            optr = o.data_ptr()
        else:
            o = np.zeros((B, L))
            optr = o.ctypes.data
        _lib.check(self._lib.rcn_cuda_features(self._h, buf.ptr, fmt, B, H, W, 1 if standardise else 0, optr))
        return o

    def gen_scales(self, feats) -> Tuple[float, float]:
        """rcn.rs:230-251: mean / population sd over all features of all samples; stored as ``scale_set``."""
        f = _Buf(feats, np.float64)
        self._use_torch_stream(f)
        m, s = C.c_double(), C.c_double()
        _lib.check(self._lib.rcn_cuda_gen_scales(self._h, f.ptr, f.shape[1], f.shape[0], C.byref(m), C.byref(s)))
        return m.value, s.value

    def standardise(self, feats):
        """rcn.rs:407-412: returns max((v - mean) / sd, 0)."""
        if _is_torch(feats):
            f = _Buf(feats.clone(), np.float64)
            self._use_torch_stream(f)
            _lib.check(self._lib.rcn_cuda_standardise(self._h, f.ptr, f.store.numel()))
            return f.store
        o = np.array(feats, dtype=np.float64, order="C", copy=True)
        _lib.check(self._lib.rcn_cuda_standardise(self._h, o.ctypes.data, o.size))
        return o

    # -- inference --------------------------------------------------------------------------------------------
    def classify_test(self, feats):
        """rcn.rs:105-116 over a batch: (B, L) features -> (B, classes) output activations."""
        self._require_params()
        f = _Buf(feats, np.float64)
        self._use_torch_stream(f)
        B = f.shape[0]
        n_out = self._shapes[-1][0]
        if f.torch:
            import torch
            o = torch.empty((B, n_out), dtype=torch.float64, device=f.device)
            optr = o.data_ptr()
        else:
            o = np.zeros((B, n_out))
            optr = o.ctypes.data
        _lib.check(self._lib.rcn_cuda_forward(self._h, f.ptr, B, optr))
        return o

    def classify_features(self, feats):
        """argmax (last maximal element wins, rcn.rs:92-97) of classify_test."""
        self._require_params()
        f = _Buf(feats, np.float64)
        self._use_torch_stream(f)
        B = f.shape[0]
        if f.torch:
            import torch
            o = torch.empty((B,), dtype=torch.int64, device=f.device)
            optr = o.data_ptr()
        else:
            o = np.zeros(B, dtype=np.int64)
            optr = o.ctypes.data
        _lib.check(self._lib.rcn_cuda_classify_features(self._h, f.ptr, B, optr))
        return o

    def classify_images(self, images):
        """``classify`` (rcn.rs:82-98) over a batch of decoded grayscale images -> class indices."""
        buf, fmt, (B, H, W) = self._images(images)
        self._use_torch_stream(buf)
        if buf.torch:
            import torch
            o = torch.empty((B,), dtype=torch.int64, device=buf.device)
            optr = o.data_ptr()
        else:
            o = np.zeros(B, dtype=np.int64)
            optr = o.ctypes.data
        _lib.check(self._lib.rcn_cuda_classify(self._h, buf.ptr, fmt, B, H, W, optr))
        return o

    def classify(self, img_path: str) -> int:
        """``RCN::classify`` (rcn.rs:82-98): open, grayscale, features, standardise, forward, argmax."""
        from .data import load_grayscale
        img = load_grayscale(img_path)
        return int(self.classify_images(img[None, :, :])[0])

    def evaluate(self, feats, labels) -> int:
        """Epoch evaluation rule (rcn.rs:152-157): number of samples whose max set equals the one-hot exactly."""
        self._require_params()
        f = _Buf(feats, np.float64)
        l = _Buf(labels, np.int64)
        self._use_torch_stream(f, l)
        acc = C.c_uint64()
        _lib.check(self._lib.rcn_cuda_evaluate(self._h, f.ptr, l.ptr, f.shape[0], C.byref(acc)))
        return acc.value

    def evaluate_images(self, images, labels, want_labels: bool = False):
        """Test-set evaluation (rcn.rs:152-157) of a batch of decoded grayscale images, standardised with ``scale_set``:
        ``(accept, cost)`` -- the exact-one-hot hit count of ``evaluate`` and the quadratic cost sum_b 0.5*|a - y|^2 --
        and with ``want_labels`` also the ``classify_images`` labels, ``(accept, cost, labels)``."""
        self._require_params()
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        cost, acc = C.c_double(), C.c_uint64()
        o, optr = None, None
        if want_labels:
            if buf.torch:
                import torch
                o = torch.empty((B,), dtype=torch.int64, device=buf.device)
                optr = o.data_ptr()
            else:
                o = np.zeros(B, dtype=np.int64)
                optr = o.ctypes.data
        _lib.check(self._lib.rcn_cuda_evaluate_images(self._h, buf.ptr, fmt, lb.ptr, B, H, W, C.addressof(cost),
                                                      C.addressof(acc), optr))
        if want_labels:
            return acc.value, cost.value, o
        return acc.value, cost.value

    # -- training ---------------------------------------------------------------------------------------------
    def _targets(self, onehot, labels):
        oh = _Buf(onehot, np.float64) if onehot is not None else None
        lb = _Buf(labels, np.int64) if labels is not None else None
        return oh, lb

    def accumulate_gradients(self, feats, onehot=None, labels=None):
        """Batch sum of backprop (rcn.rs:260-314, 190-205) into the flat gradient buffer; no update."""
        self._require_params()
        f = _Buf(feats, np.float64)
        oh, lb = self._targets(onehot, labels)
        self._use_torch_stream(f, oh, lb)
        self._B_hint = f.shape[0]
        _lib.check(self._lib.rcn_cuda_accumulate_gradients(self._h, f.ptr, oh.ptr if oh else None,
                                                           lb.ptr if lb else None, f.shape[0]))

    def accumulate_gradients_images(self, images, labels):
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        self._B_hint = B
        _lib.check(self._lib.rcn_cuda_accumulate_gradients_images(self._h, buf.ptr, fmt, lb.ptr, B, H, W))

    def apply_gradients(self, eta: float, batch: int):
        """W <- W - (eta / batch) * sum dW (rcn.rs:210-222)."""
        _lib.check(self._lib.rcn_cuda_apply_gradients(self._h, float(eta), int(batch)))

    def train_batch(self, feats, eta: float, onehot=None, labels=None):
        """``train_batch`` (rcn.rs:176-223) on (B, L) standardised features."""
        self._require_params()
        f = _Buf(feats, np.float64)
        oh, lb = self._targets(onehot, labels)
        self._use_torch_stream(f, oh, lb)
        self._B_hint = f.shape[0]
        _lib.check(self._lib.rcn_cuda_train_batch(self._h, f.ptr, oh.ptr if oh else None, lb.ptr if lb else None,
                                                  f.shape[0], float(eta)))

    def train_batch_images(self, images, labels, eta: float):
        """Features (rcn.rs:317-356) + standardise (rcn.rs:407-412) + train_batch (rcn.rs:176-223), fused on device."""
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        self._B_hint = B
        _lib.check(self._lib.rcn_cuda_train_batch_images(self._h, buf.ptr, fmt, lb.ptr, B, H, W, float(eta)))

    # -- epoch mode (rcn.rs:144-149 on a dataset resident in HBM) ---------------------------------------------------
    def epoch_bind(self, images, labels, batch: int, perm=None):
        """Bind a device-resident dataset (torch CUDA tensors): images (N, H, W) uint8, labels (N,) int64, optional
        ``perm`` (N,) int64 shuffle that may be rewritten in place between epochs. Step k then trains on samples
        ``perm[pos:pos+batch]`` with ``pos`` kept on the device (chunks_exact semantics, remainder dropped)."""
        buf, fmt, (N, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        pm = _Buf(perm, np.int64) if perm is not None else None
        if not (buf.torch and lb.torch and (pm is None or pm.torch)):
            raise ValueError("epoch mode needs torch CUDA tensors (the dataset stays resident in HBM)")
        self._use_torch_stream(buf)
        self._epoch_keepalive = (buf, lb, pm)
        self._B_hint = int(batch)
        _lib.check(self._lib.rcn_cuda_epoch_bind(self._h, buf.ptr, fmt, lb.ptr, pm.ptr if pm else None, N, H, W, int(batch)))

    def epoch_seek(self, position: int):
        _lib.check(self._lib.rcn_cuda_epoch_seek(self._h, int(position)))

    def epoch_position(self) -> int:
        p = C.c_size_t()
        _lib.check(self._lib.rcn_cuda_epoch_position(self._h, C.byref(p)))
        return p.value

    def epoch_accumulate(self):
        _lib.check(self._lib.rcn_cuda_epoch_accumulate(self._h))

    def epoch_apply(self, eta: float, global_batch: int):
        _lib.check(self._lib.rcn_cuda_epoch_apply(self._h, float(eta), int(global_batch)))

    def epoch_step(self, eta: float):
        _lib.check(self._lib.rcn_cuda_epoch_step(self._h, float(eta)))

    def epoch_run(self, eta: float, n_steps: int):
        """``n_steps`` iterations of ``for batch in training_set.chunks_exact(batch) { train_batch(batch, eta) }``
        (rcn.rs:147-149) over the bound dataset, one library call."""
        _lib.check(self._lib.rcn_cuda_epoch_run(self._h, float(eta), int(n_steps)))

    def train_epoch_host(self, images, labels, batch: int, eta: float, global_batch: int = 0):
        """``for batch in training_set.chunks_exact(batch) { train_batch(batch, eta) }`` (rcn.rs:147-149) over a HOST
        dataset (numpy, already shuffled; pin it for copy/compute overlap). The copy of chunk k+1 overlaps the kernels of
        chunk k. Returns per-step (cost, hits) arrays, read back from the device every step."""
        a = np.asarray(images)
        if a.ndim != 3:
            raise ValueError("images must be (N, H, W)")
        if a.dtype == np.uint8:
            img, fmt = np.ascontiguousarray(a), _lib.PIXELS_U8_ROWMAJOR
        else:
            img, fmt = np.ascontiguousarray(np.transpose(a, (0, 2, 1)), dtype=np.float64), _lib.PIXELS_F64_COLMAJOR
        lab = np.ascontiguousarray(labels, dtype=np.int64)
        N, H, W = a.shape
        n_steps = N // int(batch)
        cost = np.zeros(n_steps)
        hits = np.zeros(n_steps, dtype=np.uint64)
        done = C.c_size_t()
        self._B_hint = int(batch)
        _lib.check(self._lib.rcn_cuda_train_epoch_host(self._h, img.ctypes.data, fmt, lab.ctypes.data, N, H, W, int(batch),
                                                       float(eta), int(global_batch), cost.ctypes.data, hits.ctypes.data,
                                                       C.byref(done)))
        return cost[:done.value], hits[:done.value]

    # -- data-parallel group: exchange fused with the update over NVLink peer memory (csrc/dp.cu) --------------------
    def dp_init(self, world: int, rank: int) -> bytes:
        """Allocates this rank's communication block; returns its 64-byte CUDA IPC handle for the other processes."""
        buf = C.create_string_buffer(64)
        _lib.check(self._lib.rcn_cuda_dp_init(self._h, int(world), int(rank), buf))
        return buf.raw

    def dp_connect_ipc(self, handles: Sequence[bytes]):
        """handles[r] = dp_init() result of rank r (one process per GPU)."""
        blob = b"".join(handles)
        _lib.check(self._lib.rcn_cuda_dp_connect_ipc(self._h, blob))

    def dp_connect_local(self, group: Sequence["RCN"]):
        """group[r] = the RCN of rank r living in THIS process (one per device)."""
        arr = (C.c_void_p * len(group))(*[g._h.value for g in group])
        _lib.check(self._lib.rcn_cuda_dp_connect_local(self._h, arr))

    def dp_shutdown(self):
        _lib.check(self._lib.rcn_cuda_dp_shutdown(self._h))

    def timeline_enable(self, on: bool = True):
        """Device-side launch timeline of the fused step kernels (csrc/timeline.cuh); captured steps must be re-captured."""
        _lib.check(self._lib.rcn_cuda_timeline_enable(self._h, 1 if on else 0))

    def timeline_read(self):
        """(starts, ends, launches): starts / ends are (4, 64) uint64 %globaltimer ns (slot = launch index % 64) for kernel
        A, kernel B, the exchange kernel; launches (4,) uint32."""
        stamps = np.zeros((2, 4, 64), dtype=np.uint64)
        n = np.zeros(4, dtype=np.uint32)
        _lib.check(self._lib.rcn_cuda_timeline_read(self._h, stamps.ctypes.data, n.ctypes.data))
        return stamps[0], stamps[1], n

    def dp_check(self):
        """Synchronises and raises if a gradient exchange timed out waiting for a peer (the device never hangs on a dead
        or desynchronised rank: the receive is bounded, RCN_CUDA_DP_TIMEOUT_MS)."""
        e = C.c_int()
        _lib.check(self._lib.rcn_cuda_dp_error(self._h, C.byref(e)))

    def last_batch_stats(self) -> Tuple[float, int]:
        """(quadratic cost, hits) of the last accumulated batch, evaluated with the pre-update parameters."""
        c, h = C.c_double(), C.c_uint64()
        _lib.check(self._lib.rcn_cuda_last_batch_stats(self._h, C.byref(c), C.byref(h)))
        return c.value, h.value

    def activations(self, layer: int) -> np.ndarray:
        """a_{layer+1} of the last accumulated batch, (B, rows)."""
        self._require_params()
        B = self._last_B()
        buf = np.zeros((B, self._shapes[layer][0]))
        _lib.check(self._lib.rcn_cuda_get_activations(self._h, layer, buf.ctypes.data))
        return buf

    def deltas(self, layer: int) -> np.ndarray:
        self._require_params()
        B = self._last_B()
        buf = np.zeros((B, self._shapes[layer][0]))
        _lib.check(self._lib.rcn_cuda_get_deltas(self._h, layer, buf.ctypes.data))
        return buf

    def _last_B(self) -> int:
        return getattr(self, "_B_hint", 0)

    def bind_gradient_buffer(self, tensor):
        """Use a caller-owned torch CUDA float64 tensor (n_params) as the flat gradient buffer (all-reduce target)."""
        if tensor is None:
            _lib.check(self._lib.rcn_cuda_bind_gradient_buffer(self._h, None, 0))
            self._grad_keepalive = None
            return
        self._grad_keepalive = tensor
        _lib.check(self._lib.rcn_cuda_bind_gradient_buffer(self._h, tensor.data_ptr(), tensor.numel()))

    # -- whole-run driver (rcn.rs:126-167) --------------------------------------------------------------------
    def _set_stats(self, images_dev, chunk: int = 16384) -> Tuple[float, float]:
        """gen_scales (rcn.rs:230-251) over a whole device-resident set: mean / population sd of all raw features."""
        import torch
        n = images_dev.shape[0]
        if n <= chunk:
            return self.gen_scales(self.flatten_feature_set(images_dev))
        feats = torch.cat([self.flatten_feature_set(images_dev[i:i + chunk]) for i in range(0, n, chunk)])
        return self.gen_scales(feats)

    def train_arrays(self, train_images, train_labels, test_images, test_labels, batch_size: int, epochs: int,
                     eta: float, seed: int = 0, log=print, cuda_graph: bool = True):
        """``RCN::train`` (rcn.rs:126-167) on in-memory decoded images instead of PNG directories, with both sets
        RESIDENT IN HBM: scale_set from each set in turn (the training steps standardise with the training set's
        statistics, evaluation with the test set's, and scale_set ends up holding the TEST set's, rcn.rs:134-137,406);
        per-epoch shuffle (harness-seeded permutation instead of thread_rng, rewritten in place on the device);
        ``chunks_exact`` batches selected on the device by the epoch cursor (remainder dropped, rcn.rs:147); per-epoch
        evaluation with the exact-one-hot rule (rcn.rs:152-157) and the reference's log line (rcn.rs:158-164).
        Parameters must already be present (inject them with set_params) or are drawn N(0,1) from ``seed`` like
        rcn.rs:500-523. Returns the per-epoch accept counts."""
        import torch
        dev = torch.device("cuda", self.device)
        rng = np.random.default_rng(seed)
        tr = torch.as_tensor(np.ascontiguousarray(train_images)).to(dev)
        te = torch.as_tensor(np.ascontiguousarray(test_images)).to(dev)
        if tr.dtype != torch.uint8:
            tr, te = tr.to(torch.float64), te.to(torch.float64)
        tr_y = torch.as_tensor(np.asarray(train_labels, dtype=np.int64)).to(dev)
        te_y = torch.as_tensor(np.asarray(test_labels, dtype=np.int64)).to(dev)
        n, H, W = int(tr.shape[0]), int(tr.shape[1]), int(tr.shape[2])
        stream = torch.cuda.current_stream(dev)
        self.set_stream(stream.cuda_stream)
        tr_stats = self._set_stats(tr)
        te_stats = self._set_stats(te)
        if not self._shapes:
            self.load_weights_and_bias(self.feature_len(H, W))
            self.set_params(rng.standard_normal(self.n_params))
        history = []
        n_steps = n // int(batch_size)
        perm = torch.arange(n, dtype=torch.int64, device=dev)
        graph = None
        if n_steps:
            self.scale_set = tr_stats
            self.epoch_bind(tr, tr_y, int(batch_size), perm)
            if cuda_graph and tr.dtype == torch.uint8:
                side = torch.cuda.Stream(dev)
                side.wait_stream(stream)
                with torch.cuda.stream(side):
                    self.set_stream(side.cuda_stream)
                    self.epoch_accumulate()                   # warm-up launch outside capture (allocations, attributes)
                stream.wait_stream(side)

                def capture_step():
                    torch.cuda.synchronize(dev)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self.set_stream(torch.cuda.current_stream(dev).cuda_stream)
                        self.epoch_step(eta)
                    self.set_stream(stream.cuda_stream)
                    return g, _lib.allocation_generation()

                graph, graph_gen = capture_step()
        for e in range(epochs):
            if n_steps:
                perm.copy_(torch.as_tensor(rng.permutation(n)), non_blocking=False)   # training_set.shuffle (rcn.rs:146)
                self.scale_set = tr_stats
                self.epoch_seek(0)
                if graph is not None and _lib.allocation_generation() != graph_gen:
                    graph, graph_gen = capture_step()         # the evaluation below grew a library buffer: pointers moved
                for _ in range(n_steps):                      # chunks_exact(batch_size) (rcn.rs:147-149)
                    if graph is not None:
                        graph.replay()
                    else:
                        self.epoch_step(eta)
            self.scale_set = te_stats
            accept, _ = self.evaluate_images(te, te_y)
            history.append(accept)
            if log:
                log("Epoch {}: {}/{} [{:.2f}%]".format(e, accept, int(te.shape[0]), accept / max(1, int(te.shape[0])) * 100.0))
        self.scale_set = te_stats
        self.synchronize()
        return history

    def train(self, batch_size: int, epochs: int, eta: float, training_class_size_limit: int,
              testing_class_size_limit: int, seed: int = 0, log=print):
        """``RCN::train`` (rcn.rs:126-133) on the PNG class-directory trees given to the constructor."""
        from .data import load_data
        rng = np.random.default_rng(seed)
        tr_x, tr_y = load_data(self.training_path, training_class_size_limit, rng)
        te_x, te_y = load_data(self.testing_path, testing_class_size_limit, rng)
        return self.train_arrays(tr_x, tr_y, te_x, te_y, batch_size, epochs, eta, seed=seed, log=log)
