"""A trainable convolutional network: learned conv / pool layers in front of the reference's dense stack (sigmoid layers,
quadratic cost, ``W -= (eta/B) * sum dW``) or of the same stack with a softmax cross-entropy head (``Head``), driving the
``rcn_cuda_cnn_*`` entry points of librcn_cuda.so.

Images are numpy arrays (staged through the device) or torch CUDA tensors (used in place, on torch's current stream):
``(B, H, W)`` uint8 (one channel) or ``(B, H, W, C)`` float64 channels-last.  Labels are ``(B,)`` int64.  The flat
parameter and gradient layout is ``[w0 (Co,kh,kw,Ci) | b0 | w1 | b1 | ... | W0 | b0 | W1 | b1 | ...]`` -- the conv layers
in stack order, then the dense layers exactly as ``RCN.get_params`` lays them out.  The method names are the ones
``DataParallelTrainer`` calls, so the trainer's NCCL exchange drives this network unchanged.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import IntEnum
from typing import List, Sequence, Tuple

import numpy as np

from . import _lib
from .kernel import Padding, Pooling, _is_torch
from .rcn import _Buf

CNN_CONV, CNN_POOL, LAYER_INTS = 0, 1, 5


class Head(IntEnum):
    """Output head of the dense stack (``RCN_HEAD_*``, semantics in rcn_cuda.h).

    ``SigmoidQuadratic``: the reference's sigmoid output layer, cost ``sum_b 0.5 |a_b - y_b|^2``.
    ``SoftmaxCrossEntropy``: an affine output layer ``z = W a + b``, ``p = softmax(z)``, cost ``sum_b (log s + m) - z_label``
    (``m = max z``, ``s = sum exp(z - m)``) and ``delta = p - onehot(label)``; hits and labels are decided on the logits.
    Hidden layers stay sigmoid with either head."""
    SigmoidQuadratic = 0
    SoftmaxCrossEntropy = 1


@dataclass(frozen=True)
class SGD:
    """``ConvNet.set_optimizer(SGD(momentum=0.9, nesterov=False, weight_decay=5e-4))``: torch's SGD without dampening, with
    the exact operation order of rcn_cuda.h.  ``SGD()`` is the default update ``p -= (eta / B) * g``."""
    momentum: float = 0.0
    nesterov: bool = False
    weight_decay: float = 0.0


@dataclass(frozen=True)
class AdamW:
    """``ConvNet.set_optimizer(AdamW(beta1, beta2, eps, weight_decay))``: torch's AdamW with bias correction from running
    products of the betas kept on the device, with the exact operation order of rcn_cuda.h."""
    beta1: float = 0.9
    beta2: float = 0.999
    eps: float = 1e-8
    weight_decay: float = 0.0


OPTIMIZER_SGD, OPTIMIZER_ADAMW = 0, 1


@dataclass(frozen=True)
class Conv:
    """Learned cross-correlation with bias, always followed by ReLU (odd kernels for ``Padding.Same``)."""
    out_channels: int
    kh: int = 3
    kw: int = 3
    padding: Padding = Padding.Same

    def spec(self):
        return [CNN_CONV, int(self.out_channels), int(self.kh), int(self.kw), int(Padding(self.padding))]


@dataclass(frozen=True)
class Pool:
    """2x2 / stride-2 pooling; ``Padding.Same`` pads the bottom row / right column of odd maps."""
    pooling: Pooling = Pooling.Max
    padding: Padding = Padding.Same

    def spec(self):
        return [CNN_POOL, int(Pooling(self.pooling)), int(Padding(self.padding)), 0, 0]


class ConvNet:
    """``ConvNet((H, W, C), [Conv(16), Pool(), ...], feedforward=[64], classes=10, head=Head.SoftmaxCrossEntropy)``."""

    def __init__(self, input_shape: Sequence[int], layers: Sequence, feedforward: Sequence[int], classes: int, device: int = 0,
                 head: Head = Head.SigmoidQuadratic):
        self._lib = _lib.load()
        H, W, Cin = (int(x) for x in input_shape)
        self.input_shape = (H, W, Cin)
        self.layers = list(layers)
        self.feedforward = [int(x) for x in feedforward]
        self.classes = int(classes)
        self.device = int(device)
        self.head = Head(head)
        spec = [v for l in self.layers for v in l.spec()]
        arr = (C.c_int32 * max(1, len(spec)))(*spec)
        ff = (C.c_size_t * max(1, len(self.feedforward)))(*self.feedforward)
        h = C.c_void_p()
        _lib.check(self._lib.rcn_cuda_cnn_create_with_head(self.device, H, W, Cin, arr, len(self.layers), ff,
                                                           len(self.feedforward), self.classes, int(self.head), C.byref(h)))
        self._h = h
        self._shapes = []
        for i in range(len(self.layers)):
            a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
            _lib.check(self._lib.rcn_cuda_cnn_layer_shape(self._h, i, C.byref(a), C.byref(b), C.byref(c)))
            self._shapes.append((a.value, b.value, c.value))
        self._B_out = self._B_grad = 0
        self._params_set = False

    # -- lifetime -----------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.rcn_cuda_cnn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream):
        """Run on an existing cudaStream_t (int handle); ``-1`` restores the handle's own stream."""
        if cuda_stream is not None and cuda_stream < 0:
            cuda_stream = C.c_void_p(-1).value
        _lib.check(self._lib.rcn_cuda_cnn_set_stream(self._h, cuda_stream))

    def synchronize(self):
        _lib.check(self._lib.rcn_cuda_cnn_synchronize(self._h))

    def _use_torch_stream(self, *bufs):
        for b in bufs:
            if b is not None and b.torch:
                import torch
                self.set_stream(torch.cuda.current_stream(b.device).cuda_stream)
                return

    # -- shapes / parameters ------------------------------------------------------------------------------------------
    def layer_shape(self, layer: int) -> Tuple[int, int, int]:
        """(H, W, C) output of stack layer ``layer``."""
        return self._shapes[layer]

    @property
    def feature_len(self) -> int:
        h, w, c = self._shapes[-1]
        return h * w * c

    @property
    def n_params(self) -> int:
        n = C.c_size_t()
        _lib.check(self._lib.rcn_cuda_cnn_param_count(self._h, C.byref(n)))
        return n.value

    def param_slices(self) -> List[Tuple[str, slice, tuple]]:
        """(name, slice of the flat buffer, shape) of every parameter tensor, conv layers first."""
        out, off, cin = [], 0, self.input_shape[2]
        for i, l in enumerate(self.layers):
            if isinstance(l, Conv):
                shp = (l.out_channels, l.kh, l.kw, cin)
                n = int(np.prod(shp))
                out.append((f"conv{i}.w", slice(off, off + n), shp))
                off += n
                out.append((f"conv{i}.b", slice(off, off + l.out_channels), (l.out_channels,)))
                off += l.out_channels
            cin = self._shapes[i][2]
        cols = self.feature_len
        for j, rows in enumerate(self.feedforward + [self.classes]):
            out.append((f"dense{j}.W", slice(off, off + rows * cols), (rows, cols)))   # column-major rows x cols
            off += rows * cols
            out.append((f"dense{j}.b", slice(off, off + rows), (rows,)))
            off += rows
            cols = rows
        return out

    def init_params(self, rng: np.random.Generator) -> np.ndarray:
        """He-scaled N(0, 2/fan_in) conv weights, zero conv biases, and the reference's unscaled N(0, 1) for every dense
        weight and bias (rcn.rs:500-523).  Sets and returns the flat parameters."""
        p = np.zeros(self.n_params)
        for name, sl, shp in self.param_slices():
            if name.startswith("conv") and name.endswith(".w"):
                fan_in = shp[1] * shp[2] * shp[3]
                p[sl] = rng.standard_normal(sl.stop - sl.start) * np.sqrt(2.0 / fan_in)
            elif name.startswith("dense"):
                p[sl] = rng.standard_normal(sl.stop - sl.start)
        self.set_params(p)
        return p

    def set_params(self, flat):
        flat = np.ascontiguousarray(flat, dtype=np.float64).ravel()
        _lib.check(self._lib.rcn_cuda_cnn_set_params(self._h, flat.ctypes.data, flat.size))
        self._params_set = True

    def get_params(self) -> np.ndarray:
        buf = np.zeros(self.n_params)
        _lib.check(self._lib.rcn_cuda_cnn_get_params(self._h, buf.ctypes.data, buf.size))
        return buf

    def get_gradients(self) -> np.ndarray:
        buf = np.zeros(self.n_params)
        _lib.check(self._lib.rcn_cuda_cnn_get_gradients(self._h, buf.ctypes.data, buf.size))
        return buf

    # -- optimizer ------------------------------------------------------------------------------------------------------
    def set_optimizer(self, opt):
        """Selects the update of ``apply_gradients`` / ``epoch_apply`` (``SGD`` or ``AdamW``) and resets its state.  A
        captured step must be re-captured afterwards (``_lib.allocation_generation()`` changes); ``train_arrays`` and
        ``DataParallelTrainer`` do that themselves."""
        if isinstance(opt, SGD):
            args = (OPTIMIZER_SGD, float(opt.momentum), int(bool(opt.nesterov)), float(opt.weight_decay), 0.0, 0.0, 0.0)
        elif isinstance(opt, AdamW):
            args = (OPTIMIZER_ADAMW, 0.0, 0, float(opt.weight_decay), float(opt.beta1), float(opt.beta2), float(opt.eps))
        else:
            raise TypeError(f"expected SGD or AdamW, got {type(opt).__name__}")
        _lib.check(self._lib.rcn_cuda_cnn_set_optimizer(self._h, *args))

    def optimizer_state(self) -> np.ndarray:
        """The optimizer's state, flat f64: ``v`` for SGD with momentum, ``m | v | t, beta1^t, beta2^t`` for AdamW (each
        with the flat parameter layout), empty for plain SGD."""
        n = C.c_size_t()
        _lib.check(self._lib.rcn_cuda_cnn_optimizer_state_size(self._h, C.byref(n)))
        buf = np.zeros(n.value)
        _lib.check(self._lib.rcn_cuda_cnn_get_optimizer_state(self._h, buf.ctypes.data, buf.size))
        return buf

    def load_optimizer_state(self, state):
        """Restores a state from ``optimizer_state()`` of a network with the same shape and optimizer."""
        state = np.ascontiguousarray(state, dtype=np.float64).ravel()
        _lib.check(self._lib.rcn_cuda_cnn_set_optimizer_state(self._h, state.ctypes.data, state.size))

    def bind_gradient_buffer(self, tensor):
        """Use a caller-owned torch CUDA float64 tensor (n_params) as the flat gradient buffer (all-reduce target)."""
        if tensor is None:
            _lib.check(self._lib.rcn_cuda_cnn_bind_gradient_buffer(self._h, None, 0))
            self._grad_keepalive = None
            return
        self._grad_keepalive = tensor
        _lib.check(self._lib.rcn_cuda_cnn_bind_gradient_buffer(self._h, tensor.data_ptr(), tensor.numel()))

    # -- batches --------------------------------------------------------------------------------------------------------
    def _images(self, images):
        if _is_torch(images):
            import torch
            if images.dtype == torch.uint8:
                b = _Buf(images, np.uint8)
                return b, _lib.PIXELS_U8_ROWMAJOR, b.shape[:3]
            b = _Buf(images, np.float64)
            return b, _lib.PIXELS_F64_NHWC, b.shape[:3]
        a = np.asarray(images)
        if a.dtype == np.uint8:
            if a.ndim != 3:
                raise ValueError("u8 images must be (B, H, W)")
            return _Buf(a, np.uint8), _lib.PIXELS_U8_ROWMAJOR, a.shape
        if a.ndim != 4:
            raise ValueError("float images must be (B, H, W, C)")
        return _Buf(a, np.float64), _lib.PIXELS_F64_NHWC, a.shape[:3]

    def accumulate_gradients_images(self, images, labels):
        """Gradient sums of the batch into the flat gradient buffer; no update."""
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        _lib.check(self._lib.rcn_cuda_cnn_accumulate(self._h, buf.ptr, fmt, lb.ptr, B, H, W))
        self._B_out = self._B_grad = B

    def apply_gradients(self, eta: float, batch: int):
        """p <- p - (eta / batch) * g over every parameter, or the step of the optimizer set with ``set_optimizer``;
        ``batch`` is the global minibatch."""
        _lib.check(self._lib.rcn_cuda_cnn_apply(self._h, float(eta), int(batch)))

    def train_batch_images(self, images, labels, eta: float):
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        _lib.check(self._lib.rcn_cuda_cnn_train_batch(self._h, buf.ptr, fmt, lb.ptr, B, H, W, float(eta)))
        self._B_out = self._B_grad = B

    # -- epoch mode (rcn.rs:144-149 on a dataset resident in HBM) -------------------------------------------------------
    def epoch_bind(self, images, labels, batch: int, perm=None):
        """Bind a device-resident dataset (torch CUDA tensors): images (N, H, W) uint8 or (N, H, W, C) float64, labels (N,)
        int64, optional ``perm`` (N,) int64 shuffle with entries in [0, N) that may be rewritten in place between epochs.
        Step k then trains on samples ``perm[pos:pos+batch]`` with ``pos`` kept on the device (chunks_exact semantics,
        remainder dropped)."""
        buf, fmt, (N, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        pm = _Buf(perm, np.int64) if perm is not None else None
        if not (buf.torch and lb.torch and (pm is None or pm.torch)):
            raise ValueError("epoch mode needs torch CUDA tensors (the dataset stays resident in HBM)")
        self._use_torch_stream(buf)
        self._epoch_keepalive = (buf, lb, pm)
        _lib.check(self._lib.rcn_cuda_cnn_epoch_bind(self._h, buf.ptr, fmt, lb.ptr, pm.ptr if pm else None, N, H, W,
                                                     int(batch)))
        self._epoch_B = int(batch)

    def epoch_seek(self, position: int):
        _lib.check(self._lib.rcn_cuda_cnn_epoch_seek(self._h, int(position)))

    def epoch_position(self) -> int:
        p = C.c_size_t()
        _lib.check(self._lib.rcn_cuda_cnn_epoch_position(self._h, C.byref(p)))
        return p.value

    def _epoch_ran(self):
        self._B_out = self._B_grad = getattr(self, "_epoch_B", 0)

    def epoch_accumulate(self):
        """Gradient sums of the current chunk; the cursor stays."""
        _lib.check(self._lib.rcn_cuda_cnn_epoch_accumulate(self._h))
        self._epoch_ran()

    def epoch_apply(self, eta: float, global_batch: int):
        """Update with the global batch, then advance the cursor."""
        _lib.check(self._lib.rcn_cuda_cnn_epoch_apply(self._h, float(eta), int(global_batch)))

    def epoch_step(self, eta: float):
        _lib.check(self._lib.rcn_cuda_cnn_epoch_step(self._h, float(eta)))
        self._epoch_ran()

    def epoch_run(self, eta: float, n_steps: int):
        """``n_steps`` iterations of ``for batch in training_set.chunks_exact(batch) { train_batch(batch, eta) }``
        (rcn.rs:147-149) over the bound dataset, one library call."""
        _lib.check(self._lib.rcn_cuda_cnn_epoch_run(self._h, float(eta), int(n_steps)))
        if n_steps:
            self._epoch_ran()

    def train_arrays(self, train_images, train_labels, test_images, test_labels, batch_size: int, epochs: int,
                     eta: float, seed: int = 0, log=print, cuda_graph: bool = True):
        """``RCN::train`` (rcn.rs:126-167) for this network on in-memory images, both sets RESIDENT IN HBM: per epoch a
        ``default_rng(seed)`` permutation written in place on the device, ``n // batch_size`` chunks_exact steps selected by
        the device-side cursor (replays of one captured step with ``cuda_graph``, re-captured when a library buffer moved),
        then the test set evaluated in chunks of at most ``batch_size`` (accept counts summed, costs added in chunk order)
        and the reference's log line (rcn.rs:158-164).  Parameters that were never set are drawn with ``init_params`` from
        the same generator before the first permutation.  Returns the per-epoch accept counts."""
        import torch
        dev = torch.device("cuda", self.device)
        rng = np.random.default_rng(seed)
        tr = torch.as_tensor(np.ascontiguousarray(train_images)).to(dev)
        te = torch.as_tensor(np.ascontiguousarray(test_images)).to(dev)
        if tr.dtype != torch.uint8:
            tr, te = tr.to(torch.float64), te.to(torch.float64)
        tr_y = torch.as_tensor(np.asarray(train_labels, dtype=np.int64)).to(dev)
        te_y = torch.as_tensor(np.asarray(test_labels, dtype=np.int64)).to(dev)
        n, n_test, bs = int(tr.shape[0]), int(te.shape[0]), int(batch_size)
        stream = torch.cuda.current_stream(dev)
        self.set_stream(stream.cuda_stream)
        if not self._params_set:
            self.init_params(rng)
        history = []
        n_steps = n // bs
        perm = torch.arange(n, dtype=torch.int64, device=dev)
        graph = None
        if n_steps:
            self.epoch_bind(tr, tr_y, bs, perm)
            if cuda_graph:
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
                self.epoch_seek(0)
                if graph is not None and _lib.allocation_generation() != graph_gen:
                    graph, graph_gen = capture_step()         # a library buffer moved since the capture
                for _ in range(n_steps):                      # chunks_exact(batch_size) (rcn.rs:147-149)
                    if graph is not None:
                        graph.replay()
                    else:
                        self.epoch_step(eta)
                self._epoch_ran()
            accept = 0
            for i in range(0, n_test, max(1, bs)):            # never more images than a training step: no buffer grows
                a, _ = self.evaluate_images(te[i:i + bs], te_y[i:i + bs])
                accept += a
            history.append(accept)
            if log:
                log("Epoch {}: {}/{} [{:.2f}%]".format(e, accept, n_test, accept / max(1, n_test) * 100.0))
        self.synchronize()
        return history

    def last_batch_stats(self) -> Tuple[float, int]:
        """(cost, hits) of the last accumulated batch under the head's cost and hit rule, evaluated with the pre-update
        parameters."""
        c, h = C.c_double(), C.c_uint64()
        _lib.check(self._lib.rcn_cuda_cnn_last_batch_stats(self._h, C.byref(c), C.byref(h)))
        return c.value, h.value

    def _labels_out(self, buf, B):
        if buf.torch:
            import torch
            o = torch.empty((B,), dtype=torch.int64, device=buf.device)
            return o, o.data_ptr()
        o = np.zeros(B, dtype=np.int64)
        return o, o.ctypes.data

    def evaluate_images(self, images, labels, want_labels: bool = False):
        """``(accept, cost)`` of a labelled batch -- the hit count and the batch cost under the head's rules (the
        sigmoid head's are rcn.rs:153-157 and the quadratic cost) -- and with ``want_labels`` also the predicted labels,
        ``(accept, cost, labels)``.  Leaves the gradients untouched."""
        buf, fmt, (B, H, W) = self._images(images)
        lb = _Buf(labels, np.int64)
        self._use_torch_stream(buf, lb)
        cost, acc = C.c_double(), C.c_uint64()
        o, optr = self._labels_out(buf, B) if want_labels else (None, None)
        _lib.check(self._lib.rcn_cuda_cnn_evaluate_images(self._h, buf.ptr, fmt, lb.ptr, B, H, W, C.addressof(cost),
                                                          C.addressof(acc), optr))
        if B:
            self._B_out = B
        return (acc.value, cost.value, o) if want_labels else (acc.value, cost.value)

    def classify_images(self, images):
        buf, fmt, (B, H, W) = self._images(images)
        self._use_torch_stream(buf)
        o, optr = self._labels_out(buf, B)
        _lib.check(self._lib.rcn_cuda_cnn_classify_images(self._h, buf.ptr, fmt, B, H, W, optr))
        if B:
            self._B_out = B
        return o

    # -- taps -----------------------------------------------------------------------------------------------------------
    def layer_output(self, layer: int) -> np.ndarray:
        """Output of stack layer ``layer`` of the last batch run through the network, (B, H, W, C)."""
        out = np.zeros((self._B_out,) + tuple(self._shapes[layer]))
        _lib.check(self._lib.rcn_cuda_cnn_get_layer_output(self._h, int(layer), out.ctypes.data))
        return out

    def input_gradient(self) -> np.ndarray:
        """dX = W0^T delta0 of the last accumulate: (B, L), sample b's gradient with respect to its flattened features."""
        out = np.zeros((self._B_grad, self.feature_len))
        _lib.check(self._lib.rcn_cuda_cnn_get_input_gradient(self._h, out.ctypes.data))
        return out
