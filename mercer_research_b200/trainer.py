"""Data-parallel trainer: the B200 equivalent of rcn's only parallelism strategy, the per-minibatch gradient sum
over worker threads (rcn/src/rcn.rs:190-205), scaled from host threads to the GPUs of one box.

One process per GPU (torch.distributed, NCCL over NVLink 5 / NVSwitch). Every rank holds a full parameter replica,
runs features + forward + backward on its contiguous shard of the global minibatch, producing gradient SUMS in one
flat f64 buffer [dW0|db0|dW1|db1|...]; ONE all-reduce(sum) of that buffer per step; every replica then applies the
identical ``W -= (eta / B_global) * g`` (rcn.rs:210-222), so replicas stay bit-identical to each other and differ from
the single-GPU result only by summation order (SURVEY.md 8e). No other collective is on the data path.

The compute backend is any object with ``n_params``, ``bind_gradient_buffer(t)``, ``accumulate_gradients_images``,
``accumulate_gradients``, ``apply_gradients`` and ``last_batch_stats`` (``evaluate`` also needs ``evaluate_images``) --
in the product that is ``RCN`` (CUDA) or ``ConvNet`` (CUDA, NCCL exchange only);
the gloo CPU tests plug in a checker-backed stand-in to exercise exactly this host logic without a GPU.

Stream discipline: the library launches on the stream bound with ``set_stream``; the NCCL collective is ordered against
torch's CURRENT stream. Every accumulate / all-reduce / apply sequence therefore starts by binding the model to torch's
current stream (``_bind_stream``), whatever the inputs are (torch tensors, numpy arrays, pinned host buffers) -- kernels,
collective and update are then ordered by ONE stream.
"""
from __future__ import annotations

from typing import Tuple


def shard_bounds(global_batch: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of a global minibatch; the global batch must divide evenly (all BASELINE configs do)."""
    if global_batch % world:
        raise ValueError(f"global batch {global_batch} is not divisible by world size {world}")
    per = global_batch // world
    return rank * per, (rank + 1) * per


# One-shot exchange over NVLink peer memory (csrc/dp.cu) is used while every rank pushes at most this many bytes per
# step; above it the exchange is bandwidth-bound and NCCL's all-reduce (ring / NVLS in-switch reduction) wins.
P2P_MAX_PUSH_BYTES = 16 << 20


class DataParallelTrainer:
    """``exchange``: "auto" (fused NVLink peer-memory kernel for small gradient buffers, NCCL otherwise), "p2p", "nccl"."""

    def __init__(self, model, eta: float, device=None, group=None, exchange: str = "auto"):
        import torch
        import torch.distributed as dist
        self.model = model
        self.eta = float(eta)
        self.group = group
        self.dist = dist if dist.is_available() and dist.is_initialized() else None
        self.world = self.dist.get_world_size(group) if self.dist else 1
        self.rank = self.dist.get_rank(group) if self.dist else 0
        if device is None:
            device = torch.device("cuda", model.device)
        self.device = device
        # the all-reduce target IS the kernels' output buffer: no staging copy on either side of the collective
        self.grads = torch.zeros(model.n_params, dtype=torch.float64, device=device)
        model.bind_gradient_buffer(self.grads)
        self.p2p = False
        if self.world > 1 and exchange != "nccl" and hasattr(model, "dp_init") and device.type == "cuda":
            small = model.n_params * 8 * (self.world - 1) <= P2P_MAX_PUSH_BYTES
            if exchange == "p2p" or small:
                mine = model.dp_init(self.world, self.rank)          # 64-byte CUDA IPC handle of this rank's block
                handles = [None] * self.world
                self.dist.all_gather_object(handles, mine, group=group)
                model.dp_connect_ipc(handles)
                self.dist.barrier(group=group)
                self.p2p = True

    # -- plumbing ------------------------------------------------------------------------------------------------------
    def _bind_stream(self):
        """Library kernels, the NCCL all-reduce and the update all go to torch's current stream."""
        if self.device.type != "cuda" or not hasattr(self.model, "set_stream"):
            return
        import torch
        self.model.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def _same_on_all_ranks(self, value: int, what: str,
                           rule: str = "every rank must run the same number of steps per epoch"):
        """Every rank must run the same number of exchanges: a rank with fewer steps would leave its peers waiting for
        gradients that never come (the peer-memory receive would time out, the NCCL all-reduce would hang)."""
        if self.world == 1:
            return
        import torch
        dev = self.device if self.device.type == "cuda" else torch.device("cpu")
        t = torch.tensor([int(value), -int(value)], dtype=torch.int64, device=dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN, group=self.group)
        lo, hi = int(t[0].item()), -int(t[1].item())
        if lo != hi:
            raise ValueError(f"{what} differs across ranks (min {lo}, max {hi}; this rank {int(value)}): {rule}")

    def check(self):
        """Synchronises; raises if a peer-memory exchange timed out (dead or desynchronised rank)."""
        if self.p2p:
            self.model.dp_check()

    # -- one step of rcn.rs:176-223 on this rank's shard ------------------------------------------------------------
    def _reduce_and_apply(self, local_batch: int):
        if self.world > 1 and not self.p2p:
            self.dist.all_reduce(self.grads, op=self.dist.ReduceOp.SUM, group=self.group)
        self.model.apply_gradients(self.eta, local_batch * self.world)   # p2p: exchange fused into this kernel

    def step_images(self, images, labels):
        """images: this rank's shard, (B_local, H, W) uint8 / float64 (torch CUDA tensor or numpy); labels (B_local,)."""
        self._bind_stream()
        if self.world == 1 or self.p2p:   # one call: the library folds the (exchange +) update into the weight-gradient kernel
            self.model.train_batch_images(images, labels, self.eta)
            return
        self.model.accumulate_gradients_images(images, labels)
        self._reduce_and_apply(int(images.shape[0]))

    def step_features(self, feats, labels=None, onehot=None):
        self._bind_stream()
        self.model.accumulate_gradients(feats, onehot=onehot, labels=labels)
        self._reduce_and_apply(int(feats.shape[0]))

    def step_images_host(self, images, labels):
        """End-to-end step from HOST buffers (numpy, ideally pinned): H2D of the shard inside the call, and the step's
        metric (quadratic cost, hits -- evaluated with the pre-update parameters) read back from the device."""
        self._bind_stream()
        self.model.accumulate_gradients_images(images, labels)
        self._reduce_and_apply(int(images.shape[0]))
        return self.model.last_batch_stats()

    def train_epoch_host(self, images, labels, batch: int, verify_steps: bool = True):
        """This rank's shard of a host-resident dataset walked in ``chunks_exact(batch)`` steps (rcn.rs:147-149) with the
        H2D copy of the next chunk overlapping the current step; returns per-step (cost, hits) of this rank's shard.
        With the NCCL exchange the loop is driven step by step from here (the collective is a host call).
        ``verify_steps``: agree on the step count across ranks first (one small collective + a host sync); a caller that
        repeats an epoch shape every rank has already agreed on may pass False on ALL ranks."""
        n_steps = int(images.shape[0]) // int(batch)
        if verify_steps:
            self._same_on_all_ranks(n_steps, "the number of chunks_exact steps of this epoch")
        self._bind_stream()
        if self.world == 1 or self.p2p:
            return self.model.train_epoch_host(images, labels, batch, self.eta, batch * self.world)
        import numpy as np
        cost, hits = np.zeros(n_steps), np.zeros(n_steps, dtype=np.uint64)
        for k in range(n_steps):
            cost[k], hits[k] = self.step_images_host(images[k * batch:(k + 1) * batch], labels[k * batch:(k + 1) * batch])
        return cost, hits

    def step_global_images(self, images, labels):
        """Convenience: every rank passes the same GLOBAL batch and trains on its own contiguous shard of it."""
        lo, hi = shard_bounds(int(images.shape[0]), self.rank, self.world)
        self.step_images(images[lo:hi], labels[lo:hi])

    def evaluate(self, images, labels) -> Tuple[int, float]:
        """Test-set evaluation (rcn.rs:152-157) across the group: every rank passes the same GLOBAL set and evaluates a
        contiguous near-equal shard of it (the first ``n % world`` ranks take one sample more; a shard may be empty).
        Returns ``(accept, cost)`` of the whole set, identical on every rank: the hit counts are all-reduced, the costs
        gathered and added in rank order."""
        n = int(images.shape[0])
        self._same_on_all_ranks(n, "the evaluation set size", "every rank must pass the same global set")
        per, extra = divmod(n, self.world)
        lo = self.rank * per + min(self.rank, extra)
        hi = lo + per + (1 if self.rank < extra else 0)
        self._bind_stream()
        accept, cost = self.model.evaluate_images(images[lo:hi], labels[lo:hi])
        if self.world == 1:
            return int(accept), float(cost)
        import torch
        dev = self.device if self.device.type == "cuda" else torch.device("cpu")
        acc = torch.tensor([int(accept)], dtype=torch.int64, device=dev)
        self.dist.all_reduce(acc, op=self.dist.ReduceOp.SUM, group=self.group)
        mine = torch.tensor([float(cost)], dtype=torch.float64, device=dev)
        costs = [torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(costs, mine, group=self.group)
        total = 0.0
        for c in costs:          # rank order: every rank adds the same values in the same order
            total += float(c.item())
        return int(acc.item()), total

    # -- epoch mode: device-resident dataset, device-side batch cursor, one CUDA graph per step shape ---------------
    def bind_dataset(self, images, labels, batch: int, perm=None):
        """This rank's dataset shard (torch CUDA tensors). ``batch`` is the per-rank minibatch."""
        self._same_on_all_ranks(int(images.shape[0]) // int(batch), "the number of chunks_exact steps per epoch")
        self._bind_stream()
        self.model.epoch_bind(images, labels, batch, perm)
        self.local_batch = int(batch)
        self.graph = None

    def _epoch_step_eager(self):
        self._bind_stream()
        if self.world == 1 or self.p2p:   # one call: the library folds the (exchange +) update into the weight-gradient kernel
            self.model.epoch_step(self.eta)
            return
        self.model.epoch_accumulate()
        self.dist.all_reduce(self.grads, op=self.dist.ReduceOp.SUM, group=self.group)
        self.model.epoch_apply(self.eta, self.local_batch * self.world)

    def capture(self, warmup: int = 3, steps_per_graph: int = 1):
        """Captures ``steps_per_graph`` consecutive epoch steps (kernels + the NCCL all-reduce) into ONE CUDA graph; later
        epoch_step() / epoch_steps() calls replay it. The batch selection lives in device memory, so the same graph serves
        every step of every epoch; several steps per graph take the host's per-launch cost off steps that are only a few
        tens of microseconds long.

        The warm-up (buffer sizing, kernel attributes, NCCL channel set-up) runs ``warmup`` real steps on a side stream and
        then RESTORES parameters, cursor and optimizer state (momentum, AdamW's moments and step count; a model without
        ``optimizer_state`` has none): capture() leaves the training state exactly as it found it, so the step-for-step
        sequence of rcn.rs:144-149 is not advanced by it."""
        import torch
        position = self.model.epoch_position()
        params = self.model.get_params()
        opt_state = self.model.optimizer_state() if hasattr(self.model, "optimizer_state") else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._epoch_step_eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.check()
        self.model.set_params(params)
        if opt_state is not None:
            self.model.load_optimizer_state(opt_state)
        self.model.epoch_seek(position)
        self.steps_per_graph = max(1, int(steps_per_graph))
        self._capture_graph()
        return self.graph

    def _capture_graph(self):
        """Captures ``steps_per_graph`` steps without executing any (capture does not run the kernels, and the cursor and
        the parameters live in device memory): used by capture() after its warm-up and by _replay() when a library buffer
        has moved since (some call in between needed more scratch: the old graph holds freed pointers)."""
        import torch
        from . import _lib
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(self.steps_per_graph):
                self._epoch_step_eager()
        self.graph = graph
        self._graph_generation = _lib.allocation_generation()
        # (mean, sd) travel by value in the captured kernel arguments; a ConvNet has no scale_set
        self._graph_scale = getattr(self.model, "scale_set", None)
        self._bind_stream()

    def _replay(self):
        from . import _lib
        if (_lib.allocation_generation() != self._graph_generation
                or getattr(self.model, "scale_set", None) != self._graph_scale):
            self._capture_graph()
        self.graph.replay()

    def epoch_step(self):
        """One step (eager), or one replay of the captured graph (= ``steps_per_graph`` steps)."""
        if getattr(self, "graph", None) is not None:
            self._replay()
        else:
            self._epoch_step_eager()

    def epoch_steps(self, n: int):
        """Exactly ``n`` steps: whole graph replays, the remainder eagerly."""
        spg = getattr(self, "steps_per_graph", 1) if getattr(self, "graph", None) is not None else 0
        if spg:
            for _ in range(n // spg):
                self._replay()
            n -= (n // spg) * spg
        for _ in range(n):
            self._epoch_step_eager()

    def describe(self) -> str:
        if self.world == 1:
            ar = ("none (1 GPU) -> SGD update (narrow networks: applied by the weight-gradient kernel itself, "
                  "no separate launch)")
        elif self.p2p:
            ar = (f"gradient exchange of {self.model.n_params} f64 over NVLink peer memory + SGD update (narrow networks: pushed "
                  "from the weight-gradient kernel's epilogue, received + rank-ordered sum + update in one small kernel under "
                  "which the next step's front end already runs; otherwise one exchange+update kernel)")
        else:
            ar = f"1x NCCL all-reduce(sum) of {self.model.n_params} f64 per step -> SGD update"
        return ("features(+standardise) -> fwd -> bwd-data -> bwd-weight(+db) -> batch stats -> " + ar +
                "; kernels launched through the C ABI on torch's current stream")
