"""World-size-2/3 CPU (gloo) test of the class-sharded head with the focal loss: the host logic
of tf_face_toolbox_b200/sharded.py (collectives, statistics exchange, dX reduce-scatter) driving
an injected float64 shard built on oracle/focal_ref.py's class-sharded form.  Every rank must
report the same loss, and the gathered dX and dW must equal the one-piece focal oracle."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import focal_ref as fr
from tf_face_toolbox_b200 import FocalLoss
from tf_face_toolbox_b200.sharded import ShardedASoftmaxHead, shard_bounds
from tf_face_toolbox_b200.synthetic import make_inputs

GAMMA, ALPHA, LAM = 0.7, 2.0, 5.0


class FocalOracleShard:
    """forward_partial / backward_partial with the C ABI's semantics under asm_set_loss(FOCAL)."""

    def __init__(self, lo, hi, m, loss):
        self.lo, self.hi, self.m, self.loss = lo, hi, m, loss

    def forward_partial(self, X, y, W, lam):
        self.X, self.y, self.W, self.lam = X.double().numpy(), y.numpy(), W.double().numpy(), lam
        mloc, zloc, fy, _ = fr.sharded_partial_stats(self.X, self.W, self.y, self.lo, self.m, lam)
        return torch.from_numpy(np.stack([mloc, zloc, fy])).float()

    def backward_partial(self, stats_all, X, W):
        st = stats_all.double().numpy()
        M, logZ, w, loss = fr.sharded_combine([(st[g, 0], st[g, 1], st[g, 2]) for g in range(st.shape[0])],
                                              self.loss.gamma, self.loss.alpha)
        dXp, dW = fr.sharded_backward(self.X, self.W, self.y, self.lo, M, logZ, w, self.m, self.lam)
        return torch.tensor(loss, dtype=torch.float32), torch.from_numpy(dXp).float(), torch.from_numpy(dW).float()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, B, D, Cn, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        inp = make_inputs(B, D, Cn, seed=5, w_std=0.05)
        lo, hi = shard_bounds(Cn, world, rank)
        loss_kind = FocalLoss(GAMMA, ALPHA)
        head = ShardedASoftmaxHead(D, Cn, m=4, mode="fp32", device="cpu", weights_full=inp.W, loss=loss_kind,
                                   shard_compute=FocalOracleShard(lo, hi, 4, loss_kind))
        assert head.loss == loss_kind
        b = B // world
        loss, dX_local, dW_local = head.step(inp.X[rank * b:(rank + 1) * b], inp.y[rank * b:(rank + 1) * b], LAM)
        q.put((rank, float(loss), dX_local.numpy(), dW_local.numpy(), lo, hi))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_focal_step_equals_one_piece_oracle(world):
    B, D, Cn = 12, 16, 37
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, B, D, Cn, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = sorted([q.get(timeout=120) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    inp = make_inputs(B, D, Cn, seed=5, w_std=0.05)
    full = fr.focal_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), GAMMA, ALPHA, 4, LAM)
    assert len({o[1] for o in outs}) == 1                      # the same loss on every rank
    b = B // world
    dX = np.concatenate([o[2] for o in outs])
    dW = np.concatenate([o[3] for o in outs], axis=1)
    assert outs[0][1] == pytest.approx(full.loss, rel=1e-6)
    np.testing.assert_allclose(dX, full.dX, rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(dW, full.dW, rtol=1e-4, atol=1e-7)
    assert dX.shape == (world * b, D) and dW.shape == (D, Cn)
