"""CPU (gloo, world_size 2) tests of DataParallelTrainer.evaluate: every rank passes the same global set, evaluates a
contiguous near-equal shard (the first n % world ranks take one sample more, a shard may be empty), and every rank
returns the accept count and cost of the whole set.  The per-shard evaluation here is the oracle; on a GPU box it is
RCN.evaluate_images."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = [1, 3]
SHAPES = [(30, 784), (10, 30)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def oracle_evaluate(params, mean, sd, images, labels):
    """(accept, cost) of rcn.rs:152-157 and the quadratic cost over a set."""
    import oracle as O
    images, labels = np.asarray(images), np.asarray(labels)
    if len(images) == 0:
        return 0, 0.0
    acts = O.Net(SHAPES).forward(params, O.standardise(O.features_u8(CFG, images), mean, sd))
    y = np.eye(acts.shape[1])[labels]
    return O.accuracy(acts, labels), 0.5 * float(np.sum((acts - y) ** 2))


class OracleModel:
    """What DataParallelTrainer needs of the model, computed by the CPU oracle."""

    def __init__(self, params, mean, sd):
        self.params, self.mean, self.sd = params, mean, sd
        self.n_params = len(params)
        self.device = 0
        self.shards = []

    def bind_gradient_buffer(self, t):
        pass

    def evaluate_images(self, images, labels):
        self.shards.append(len(images))
        return oracle_evaluate(self.params, self.mean, self.sd, images, labels)


def data(n):
    import oracle as O
    rng = np.random.default_rng(0x5EED + n)
    images = rng.integers(0, 256, size=(n, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=n).astype(np.int64)
    params = np.random.default_rng(0xC0FFEE).standard_normal(O.Net(SHAPES).n_params) * 0.1
    mean, sd = O.gen_scales(O.features_u8(CFG, rng.integers(0, 256, size=(8, 28, 28), dtype=np.uint8)))
    return images, labels, params, mean, sd


def _worker(rank, world, port, n, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from mercer_research_b200.trainer import DataParallelTrainer
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    images, labels, params, mean, sd = data(n)
    model = OracleModel(params, mean, sd)
    trainer = DataParallelTrainer(model, eta=3.0, device=torch.device("cpu"))
    acc, cost = trainer.evaluate(images, labels)
    assert isinstance(acc, int) and isinstance(cost, float)
    np.save(os.path.join(out_dir, f"eval_{rank}.npy"), np.array([acc, cost, model.shards[0]], dtype=np.float64))
    dist.destroy_process_group()


@pytest.mark.parametrize("n, shards", [(17, [9, 8]), (1, [1, 0])])
def test_evaluate_two_ranks_equals_single_process(tmp_path, n, shards):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), n, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "eval_0.npy"), np.load(tmp_path / "eval_1.npy")
    assert [int(r0[2]), int(r1[2])] == shards
    assert np.array_equal(r0[:2], r1[:2]), "every rank must return the same values"
    images, labels, params, mean, sd = data(n)
    acc, cost = oracle_evaluate(params, mean, sd, images, labels)
    assert int(r0[0]) == acc
    assert abs(r0[1] - cost) <= 1e-12 * abs(cost)
