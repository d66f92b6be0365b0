"""GPU parity tests: the CUDA path (through the C ABI) against the float64 oracle.

Tolerances are BASELINE.json's: exact label / argmax indexing, loss within 1e-5 relative
(fp32 mode) / 2e-3 relative (bf16 mode), gradient cosine similarity >= 0.9999.
"""
import os

import numpy as np
import pytest
import torch

from head_checks import LOSS_TOL, assert_within_oracle_bounds, check_fused_optimizer_against_unfused, cosine
from oracle import asoftmax_ref as ref
from tf_face_toolbox_b200 import ASoftmaxHead, ASoftmaxLoss, LambdaState, asoftmax_head
from tf_face_toolbox_b200 import _lib
from tf_face_toolbox_b200.synthetic import make_inputs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def run_gpu(inp, m, lam, mode, return_logits=False):
    dev = torch.device("cuda:0")
    loss, logits, dX, dW = asoftmax_head(inp.X.to(dev), inp.y.to(dev), inp.W.shape[1], m, lam,
                                         weights=inp.W.to(dev), mode=mode, return_logits=return_logits,
                                         check_labels=True)
    torch.cuda.synchronize()
    return (float(loss), None if logits is None else logits.cpu().numpy(), dX.cpu().numpy(), dW.cpu().numpy())


def check_against_oracle(inp, m, lam, mode, logits=False, cos_min=0.9999, loss_floor=0.0):
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), m, lam)
    loss, f, dX, dW = run_gpu(inp, m, lam, mode, return_logits=logits)
    assert_within_oracle_bounds(inp, r, mode, loss, f, dX, dW, cos_min=cos_min, loss_floor=loss_floor)
    return loss, dX, dW, r


# ------------------------------------------------------------------------- fp32 mode
@pytest.mark.parametrize("B,D,C", [(37, 64, 1000), (5, 16, 7), (130, 48, 1001), (256, 128, 2049)])
@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_fp32_small_shapes_all_margins(B, D, C, m):
    inp = make_inputs(B, D, C, seed=100 + m, w_std=0.05)
    check_against_oracle(inp, m, 5.0, "fp32", logits=True)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,D,C", [(1, 64, 300), (32, 64, 5), (256, 1024, 2000), (64, 2048, 1500), (700, 256, 1300)])
def test_edge_shapes_on_the_tensor_core_kernels(B, D, C, mode):
    """One row, fewer classes than a tile, wide embeddings (the reference's ResNeXt emits
    D = 2048, nets/resnext.py), a batch that is not a multiple of the 128-row tile."""
    inp = make_inputs(B, D, C, seed=77)
    check_against_oracle(inp, 4, 5.0, mode, loss_floor=10.0 if B == 1 else 0.0)


@pytest.mark.parametrize("lam", [0.0, 5.0, 1000 / 1.12])
def test_fp32_lambda_values(lam):
    inp = make_inputs(64, 128, 3000, seed=5)
    check_against_oracle(inp, 4, lam, "fp32", logits=True)


def test_fp32_cfg1_full_size():
    """BASELINE config 1: head alone, m=4, D=512, C=10,572, batch 256, fp32."""
    inp = make_inputs(256, 512, 10572)
    check_against_oracle(inp, 4, 5.0, "fp32", logits=True)


@pytest.mark.parametrize("B,D,C", [(64, 64, 300), (256, 512, 10572)])
def test_fp32_cuda_core_kernels_still_match(B, D, C, monkeypatch):
    """ASM_FP32_SIMT=1 selects the CUDA-core fp32 kernels for shapes the tcgen05 path covers."""
    monkeypatch.setenv("ASM_FP32_SIMT", "1")
    dev = torch.device("cuda:0")
    inp = make_inputs(B, D, C, seed=5)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    loss, _, dX, dW = asoftmax_head(inp.X.to(dev), inp.y.to(dev), C, 4, 5.0, weights=inp.W.to(dev),
                                    mode="fp32", _handle_tag="simt")
    assert abs(float(loss) - r.loss) <= 1e-5 * abs(r.loss)
    np.testing.assert_allclose(dX.cpu().numpy(), r.dX, rtol=2e-3, atol=1e-6 * np.abs(r.dX).max() + 1e-12)
    np.testing.assert_allclose(dW.cpu().numpy(), r.dW, rtol=2e-3, atol=1e-5 * np.abs(r.dW).max() + 1e-12)


def test_fp32_golden_fixtures_through_c_abi():
    z = np.load(os.path.join(GOLD, "asoftmax_small.npz"))
    for key in [k[:-5] for k in z.files if k.endswith("_loss")]:
        B, D, C, m = (int(v) for v in z[key + "_shape"])
        lam = float(z[key + "_lam"])
        inp = make_inputs(B, D, C, seed=int(z[key + "_seed"]), w_std=0.05)
        loss, f, dX, dW = run_gpu(inp, m, lam, "fp32", return_logits=True)
        assert abs(loss - float(z[key + "_loss"])) <= 1e-5 * abs(float(z[key + "_loss"]))
        assert cosine(dX, z[key + "_dX"]) >= 0.99999
        assert cosine(dW, z[key + "_dW"]) >= 0.99999
        np.testing.assert_allclose(f, z[key + "_logits"], atol=2e-5, rtol=1e-4)


# ------------------------------------------------------------------------- bf16 mode
@pytest.mark.parametrize("B,D,C", [(128, 64, 256), (100, 128, 1000), (512, 512, 10572), (300, 192, 777)])
def test_bf16_shapes(B, D, C):
    inp = make_inputs(B, D, C, seed=21)
    check_against_oracle(inp, 4, 5.0, "bf16", logits=True)


@pytest.mark.parametrize("m,lam", [(1, 0.0), (2, 1.0), (3, 5.0), (4, 0.0), (4, 1000 / 1.12)])
def test_bf16_margins_and_lambdas(m, lam):
    inp = make_inputs(256, 512, 4000, seed=31)
    check_against_oracle(inp, m, lam, "bf16")


def test_bf16_matches_fp32_path_on_device():
    inp = make_inputs(512, 512, 10572, seed=3)
    l32, _, dX32, dW32 = run_gpu(inp, 4, 5.0, "fp32")
    l16, _, dX16, dW16 = run_gpu(inp, 4, 5.0, "bf16")
    assert abs(l16 - l32) <= 2e-3 * abs(l32)
    assert cosine(dX16, dX32) >= 0.9999
    assert cosine(dW16, dW32) >= 0.9999


def test_bf16_cfg3_full_size_vs_oracle_and_properties():
    """BASELINE config 3 (the metric): C=85,742, D=512, batch 512, bf16 -- against the oracle
    and through size-independent properties (dW_j orthogonal to w_j, column-scale invariance)."""
    inp = make_inputs(512, 512, 85742)
    loss, dX, dW, r = check_against_oracle(inp, 4, 5.0, "bf16")
    W = inp.W.double().numpy()
    # normalisation Jacobian: dW_j . w_j = 0 (relative to |dW_j||w_j|)
    num = np.abs((dW.astype(np.float64) * W).sum(axis=0))
    den = np.sqrt((dW.astype(np.float64) ** 2).sum(axis=0) * (W ** 2).sum(axis=0)) + 1e-30
    assert np.median(num / den) < 2e-2
    # scale invariance: W * diag(alpha) leaves loss and dX unchanged, dW columns scale by 1/alpha
    g = torch.Generator().manual_seed(9)
    alpha = torch.exp2(torch.randint(-2, 3, (85742,), generator=g).float())   # powers of two: exact in bf16
    inp2 = type(inp)(inp.X, (inp.W * alpha).contiguous(), inp.y)
    loss2, _, dX2, dW2 = run_gpu(inp2, 4, 5.0, "bf16")
    assert abs(loss2 - loss) <= 1e-5 * abs(loss)
    assert cosine(dX2, dX) >= 0.999999
    assert cosine(dW2 * alpha.numpy(), dW) >= 0.999999


# ------------------------------------------------------------------------- interface
def test_forward_only_and_logits_null_path():
    inp = make_inputs(64, 128, 3000, seed=5)
    dev = torch.device("cuda:0")
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    loss, logits, dX, dW = asoftmax_head(inp.X.to(dev), inp.y.to(dev), 3000, 4, 5.0, weights=inp.W.to(dev),
                                         mode="fp32", compute_grads=False)
    assert logits is None and dX is None and dW is None
    assert abs(float(loss) - r.loss) <= 1e-5 * r.loss


def test_int64_labels_and_lambda_state():
    inp = make_inputs(64, 128, 3000, seed=5)
    dev = torch.device("cuda:0")
    st = LambdaState()
    st.step()
    assert st.value() == pytest.approx(1000 / 1.12)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, st.value())
    loss, *_ = asoftmax_head(inp.X.to(dev), inp.y.long().to(dev), 3000, 4, st, weights=inp.W.to(dev), mode="fp32")
    assert abs(float(loss) - r.loss) <= 1e-5 * r.loss
    assert _lib.load().asm_lambda(1, 1000.0, 0.12, 1.0, 5.0) == pytest.approx(ref.lambda_schedule(1), rel=1e-6)


def test_label_out_of_range_is_reported_not_fatal():
    inp = make_inputs(32, 64, 100, seed=5)
    dev = torch.device("cuda:0")
    y = inp.y.clone()
    y[3] = 100
    with pytest.raises(_lib.AsmError) as ei:
        asoftmax_head(inp.X.to(dev), y.to(dev), 100, 4, 5.0, weights=inp.W.to(dev), mode="fp32", check_labels=True)
    assert ei.value.code == _lib.ASM_ERR_LABEL_RANGE
    # the device is still healthy
    check_against_oracle(inp, 4, 5.0, "fp32")


def test_invalid_arguments_raise():
    inp = make_inputs(32, 64, 100, seed=5)
    dev = torch.device("cuda:0")
    with pytest.raises(RuntimeError):
        asoftmax_head(inp.X, inp.y, 100, 4, 5.0, weights=inp.W, mode="fp32")          # CPU tensors
    with pytest.raises(ValueError):
        asoftmax_head(inp.X.to(dev), inp.y.to(dev), 101, 4, 5.0, weights=inp.W.to(dev), mode="fp32")
    with pytest.raises(_lib.AsmError):
        asoftmax_head(inp.X.to(dev), inp.y.to(dev), 100, 5, 5.0, weights=inp.W.to(dev), mode="fp32")  # m=5


def test_network_shaped_wrapper_and_autograd_bridge():
    dev = torch.device("cuda:0")
    inp = make_inputs(64, 128, 500, seed=8)
    head = ASoftmaxHead(128, 500, m=4, mode="fp32", device=dev, return_logits=True)
    head.weights.copy_(inp.W.to(dev))
    out = head.forward(inp.X.to(dev), inp.y.to(dev), num_classes=500, is_training=True)
    losses, names, others = head.loss_function("TOWER_0", inp.y.to(dev), **out)
    assert names == ["cross_entropy", "reg_loss"]
    lam = ref.lambda_schedule(1)
    assert others["lambda"] == pytest.approx(lam)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, lam)
    assert abs(float(losses[0]) - r.loss) <= 1e-5 * r.loss
    assert float(losses[1]) == pytest.approx(0.5 * 5e-4 * float((inp.W ** 2).sum()), rel=1e-5)
    dX, dW = head.gradients(num_gpus=1)
    assert cosine(dX.cpu().numpy(), r.dX) >= 0.99999
    assert cosine(dW.cpu().numpy(), r.dW + 5e-4 * inp.W.numpy()) >= 0.99999
    assert head.forward(inp.X.to(dev), is_training=False) is not None
    # autograd bridge
    X = inp.X.to(dev).requires_grad_(True)
    W = inp.W.to(dev).requires_grad_(True)
    loss = ASoftmaxLoss.apply(X, W, inp.y.to(dev), 4, 5.0, "fp32")
    (2.0 * loss).backward()
    r5 = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    assert cosine(X.grad.cpu().numpy(), 2 * r5.dX) >= 0.99999
    np.testing.assert_allclose(W.grad.cpu().numpy(), 2 * r5.dW, rtol=5e-3, atol=1e-5 * np.abs(r5.dW).max())


# ------------------------------------------------------------------------- class shards
@pytest.mark.parametrize("mode,G", [("fp32", 3), ("bf16", 2), ("bf16", 8)])
def test_class_sharded_partials_equal_unsharded(mode, G):
    """Run G class shards one after another on one GPU through asm_forward_partial /
    asm_backward_partial and combine them like the collectives would."""
    import ctypes as C
    from tf_face_toolbox_b200.sharded import _CudaShard, shard_bounds
    dev = torch.device("cuda:0")
    B, D, Cn = 96, 128, 5000
    inp = make_inputs(B, D, Cn, seed=77)
    X, y = inp.X.to(dev), inp.y.to(dev)
    shards = []
    for g in range(G):
        lo, hi = shard_bounds(Cn, G, g)
        sh = _CudaShard(D, Cn, lo, hi, 4, mode, g, G, dev)
        Wg = inp.W[:, lo:hi].contiguous().to(dev)
        shards.append((sh, Wg, lo, hi))
    stats = [sh.forward_partial(X, y, Wg, 5.0) for sh, Wg, _, _ in shards]
    stats_all = torch.stack(stats).contiguous()
    dX = torch.zeros(B, D, device=dev)
    dW = torch.empty(D, Cn, device=dev)
    losses = []
    for sh, Wg, lo, hi in shards:
        loss, dXp, dWg = sh.backward_partial(stats_all, X, Wg)
        dX += dXp
        dW[:, lo:hi] = dWg
        losses.append(float(loss))
    torch.cuda.synchronize()
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    assert max(losses) - min(losses) == 0.0
    assert abs(losses[0] - r.loss) <= LOSS_TOL[mode] * r.loss
    assert cosine(dX.cpu().numpy(), r.dX) >= 0.9999
    assert cosine(dW.cpu().numpy(), r.dW) >= 0.9999


def test_repeatable_bitwise():
    inp = make_inputs(256, 512, 4000, seed=31)
    a = run_gpu(inp, 4, 5.0, "bf16")
    b = run_gpu(inp, 4, 5.0, "bf16")
    assert a[0] == b[0]
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])


def test_cuda_graph_step_matches_eager_and_follows_lambda():
    """GraphedASoftmaxStep: same results as the eager call, lambda read from device memory."""
    from tf_face_toolbox_b200 import GraphedASoftmaxStep
    dev = torch.device("cuda:0")
    inp = make_inputs(256, 512, 4000, seed=31)
    W = inp.W.to(dev)
    step = GraphedASoftmaxStep(W, batch_size=256, m=4, mode="bf16")
    for lam in (5.0, 0.0, 1000 / 1.12):
        loss_g, dX_g, dW_g = step(inp.X.pin_memory(), inp.y.pin_memory(), lam)
        torch.cuda.synchronize()
        loss_e, _, dX_e, dW_e = asoftmax_head(inp.X.to(dev), inp.y.to(dev), 4000, 4, lam, weights=W, mode="bf16")
        torch.cuda.synchronize()
        assert float(loss_g) == float(loss_e)
        assert torch.equal(dX_g, dX_e) and torch.equal(dW_g, dW_e)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 1000 / 1.12)
    assert abs(float(loss_g) - r.loss) <= 2e-3 * r.loss


@pytest.mark.parametrize("kind", ["Momentum", "Adam"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_fused_optimizer_matches_unfused_update(kind, mode):
    """§8f-1: the optimizer fused into the dW epilogue equals grad-then-update over 3 steps
    (TF Momentum / Adam semantics on cross_entropy + L2 reg_loss, data_parallel.py:186-196)."""
    check_fused_optimizer_against_unfused(kind, mode)


def test_center_loss_gpu_matches_oracle_including_duplicates_and_shards():
    """§8f-2: center loss (loss.py:29-45) on the GPU, whole and class-sharded."""
    from tf_face_toolbox_b200.center import center_loss
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(5)
    B, D, Cn = 300, 512, 40                       # many duplicate labels
    X = torch.randn(B, D, generator=g)
    y = torch.randint(0, Cn, (B,), generator=g).to(torch.int32)
    cen = torch.randn(Cn, D, generator=g) * 0.1
    loss_r, new_r, grad_r = ref.center_loss(X.numpy(), y.numpy(), cen.numpy(), alpha=0.95, weight=0.7)
    c_dev = cen.clone().to(dev)
    loss, grad = center_loss(X.to(dev), y.to(dev), c_dev, alpha=0.95, weight=0.7)
    torch.cuda.synchronize()
    assert float(loss) == pytest.approx(loss_r, rel=1e-5)
    np.testing.assert_allclose(grad.cpu().numpy(), grad_r, rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(c_dev.cpu().numpy(), new_r, rtol=1e-4, atol=1e-6)
    # two class shards: partial losses add up, gradients / updates are disjoint
    lo = 17
    cA, cB = cen[:lo].clone().to(dev), cen[lo:].clone().to(dev)
    acc = torch.zeros(B, D, device=dev)
    lA, _ = center_loss(X.to(dev), y.to(dev), cA, 0.95, 0.7, class_offset=0, grad_accum=acc)
    lB, _ = center_loss(X.to(dev), y.to(dev), cB, 0.95, 0.7, class_offset=lo, grad_accum=acc)
    torch.cuda.synchronize()
    assert float(lA) + float(lB) == pytest.approx(loss_r, rel=1e-5)
    np.testing.assert_allclose(acc.cpu().numpy(), grad_r, rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(torch.cat([cA, cB]).cpu().numpy(), new_r, rtol=1e-4, atol=1e-6)


def test_train_loop_glue_loss_decreases():
    """§8f-4: torch SphereFaceNet-20 backbone + fused-optimizer head, reference-shaped loop."""
    import importlib.util
    import sys as _sys
    spec = importlib.util.spec_from_file_location(
        "train_sphereface20", os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "train_sphereface20.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    argv = _sys.argv
    _sys.argv = ["train_sphereface20.py", "--steps", "32", "--batch", "64", "--classes", "1000", "--lr", "0.01"]
    try:
        first, last = mod.main()
    finally:
        _sys.argv = argv
    assert np.isfinite(first) and np.isfinite(last) and last < first


def test_host_pipelined_step_returns_every_loss_in_order():
    """HostPipelinedStep: async double-buffered H2D + one-step-late loss read-back gives the
    same per-step losses as the plain synchronous loop."""
    from tf_face_toolbox_b200.pipeline import HostPipelinedStep
    dev = torch.device("cuda:0")
    W = make_inputs(64, 128, 1000, seed=1).W.to(dev)
    batches = [make_inputs(64, 128, 1000, seed=100 + i) for i in range(5)]
    want = []
    for b in batches:
        loss, *_ = asoftmax_head(b.X.to(dev), b.y.to(dev), 1000, 4, 5.0, weights=W, mode="fp32")
        want.append(float(loss))
    runner = HostPipelinedStep(lambda X, y: (lambda o: (o[0], o[2], o[3]))(
        asoftmax_head(X, y, 1000, 4, 5.0, weights=W, mode="fp32")), 64, 128, dev)
    got = []
    for b in batches:
        prev = runner.submit(b.X.pin_memory(), b.y.pin_memory())
        if prev is not None:
            got.append(prev)
    got.append(runner.flush())
    assert got == want


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_sharded_head_fused_optimizer_matches_single_call(mode):
    """The class-sharded head's step(optimizer=...) (asm_forward_partial / asm_backward_partial
    with the update fused into the shard's dW kernel) equals the single-shard fused call."""
    from tf_face_toolbox_b200 import FusedOptimizer, ShardedASoftmaxHead
    dev = torch.device("cuda:0")
    inp = make_inputs(256, 128, 3000, seed=9)
    X, y = inp.X.to(dev), inp.y.to(dev)
    head = ShardedASoftmaxHead(128, 3000, m=4, mode=mode, device=dev, weights_full=inp.W)   # world 1
    W = inp.W.to(dev).clone()
    o1, o2 = FusedOptimizer("Momentum", lr=0.05), FusedOptimizer("Momentum", lr=0.05)
    for _ in range(3):
        l1, dX1, none_dW = head.step(X, y, 5.0, optimizer=o1)
        l2, _, dX2, _ = asoftmax_head(X, y, 3000, 4, 5.0, weights=W, mode=mode, optimizer=o2)
        assert none_dW is None
    torch.cuda.synchronize()
    assert float(l1) == pytest.approx(float(l2), rel=1e-6)
    torch.testing.assert_close(head.weights, W, rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(o1.state0, o2.state0, rtol=1e-5, atol=1e-10)
    torch.testing.assert_close(dX1, dX2, rtol=1e-5, atol=1e-9)
    assert not torch.equal(W, inp.W.to(dev))                      # the weights did move


# ------------------------------------------------------------------------- round 2 additions
def test_fused_optimizer_on_cuda_core_path_keeps_dx(monkeypatch):
    """ADVICE r1: with the CUDA-core fp32 kernels the dX kernel reads the fp32 weights the fused
    optimizer rewrites; dX must equal the unfused call's dX bit for bit (dX runs first there)."""
    from tf_face_toolbox_b200 import FusedOptimizer
    monkeypatch.setenv("ASM_FP32_SIMT", "1")
    dev = torch.device("cuda:0")
    B, D, Cn = 96, 128, 2000
    inp = make_inputs(B, D, Cn, seed=43)
    X, y = inp.X.to(dev), inp.y.to(dev)
    W = inp.W.to(dev)
    _, _, dX_plain, dW_plain = asoftmax_head(X, y, Cn, 4, 5.0, weights=W, mode="fp32", _handle_tag="simt-opt")
    Wf = W.clone()
    opt = FusedOptimizer("Momentum", lr=0.5, weight_decay=0.0)         # a large step: a race would show
    for _ in range(3):
        Wf.copy_(W)
        opt.state0 = None
        _, _, dX_fused, none_dW = asoftmax_head(X, y, Cn, 4, 5.0, weights=Wf, mode="fp32", optimizer=opt,
                                                _handle_tag="simt-opt")
        assert none_dW is None
        torch.cuda.synchronize()
        assert torch.equal(dX_fused, dX_plain)
    torch.testing.assert_close(Wf, W - 0.5 * dW_plain, rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_gradient_transform_and_reg_loss_cost_no_pass(mode):
    """grad_scale / weight_decay / reg_loss_out (asm_set_gradient_transform): what the towers do
    to the gradients (data_parallel.py:32-38: tf.gradients(cross_entropy + reg_loss) * mult_lr /
    num_gpus; nets/net_base.py:103-107) applied inside the kernels."""
    dev = torch.device("cuda:0")
    B, D, Cn = 192, 128, 3002                     # C % 4 == 2: the shifted odd-row dW boxes
    inp = make_inputs(B, D, Cn, seed=51)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    gs, wd = 0.125, 5e-4
    reg = torch.zeros(1, device=dev)
    loss, _, dX, dW = asoftmax_head(inp.X.to(dev), inp.y.to(dev), Cn, 4, 5.0, weights=inp.W.to(dev), mode=mode,
                                    grad_scale=gs, weight_decay=wd, reg_loss_out=reg)
    torch.cuda.synchronize()
    assert abs(float(loss) - r.loss) <= LOSS_TOL[mode] * r.loss            # the loss itself is not scaled
    assert float(reg) == pytest.approx(0.5 * wd * float((inp.W.double() ** 2).sum()), rel=1e-5)
    want_dW = gs * (r.dW + wd * inp.W.double().numpy())
    assert cosine(dX.cpu().numpy(), gs * r.dX) >= 0.9999
    assert cosine(dW.cpu().numpy(), want_dW) >= 0.9999
    tol = 2e-5 if mode == "fp32" else 2e-2
    np.testing.assert_allclose(dX.cpu().numpy(), gs * r.dX, rtol=0, atol=tol * np.abs(gs * r.dX).max())
    np.testing.assert_allclose(dW.cpu().numpy(), want_dW, rtol=0, atol=tol * np.abs(want_dW).max())
    # the handle is back to the defaults afterwards
    _, _, dX1, dW1 = asoftmax_head(inp.X.to(dev), inp.y.to(dev), Cn, 4, 5.0, weights=inp.W.to(dev), mode=mode)
    assert cosine(dW1.cpu().numpy(), r.dW) >= 0.9999 and abs(float(dX1.abs().max()) / np.abs(r.dX).max() - 1) < 0.05


def test_network_wrapper_makes_no_eager_pass_over_weights():
    """VERDICT r1 weak #10: loss_function / gradients of the Network-shaped wrapper take reg_loss
    and the scaled, weight-decayed gradients straight from the kernels."""
    dev = torch.device("cuda:0")
    inp = make_inputs(64, 128, 500, seed=8)
    head = ASoftmaxHead(128, 500, m=4, mode="fp32", device=dev, num_gpus=4, mult_lr=2.0,
                        lambda_state=LambdaState(explicit=5.0))
    head.weights.copy_(inp.W.to(dev))
    out = head.forward(inp.X.to(dev), inp.y.to(dev), num_classes=500, is_training=True)
    losses, names, _ = head.loss_function("TOWER_0", inp.y.to(dev), **out)
    dX, dW = head.gradients()
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    assert names == ["cross_entropy", "reg_loss"]
    assert float(losses[1]) == pytest.approx(0.5 * 5e-4 * float((inp.W.double() ** 2).sum()), rel=1e-5)
    np.testing.assert_allclose(dX.cpu().numpy(), 0.5 * r.dX, rtol=2e-3, atol=1e-5 * np.abs(r.dX).max())
    np.testing.assert_allclose(dW.cpu().numpy(), 0.5 * (r.dW + 5e-4 * inp.W.numpy()), rtol=2e-3,
                               atol=1e-5 * np.abs(r.dW).max())
    dX1, dW1 = head.gradients(num_gpus=1, mult_lr=1.0)             # another scale: rescaled on request
    np.testing.assert_allclose(dX1.cpu().numpy(), r.dX, rtol=2e-3, atol=1e-5 * np.abs(r.dX).max())


def test_out_of_range_label_poisons_the_loss():
    """ADVICE r1: a label outside [0, C) must not yield a finite-but-wrong loss when nobody asks
    asm_check_labels: the row's loss is NaN (as TF's sparse softmax CE yields on the GPU)."""
    inp = make_inputs(32, 64, 100, seed=5)
    dev = torch.device("cuda:0")
    y = inp.y.clone()
    y[3] = 100
    loss, *_ = asoftmax_head(inp.X.to(dev), y.to(dev), 100, 4, 5.0, weights=inp.W.to(dev), mode="fp32")
    assert np.isnan(float(loss))
    loss, *_ = asoftmax_head(inp.X.to(dev), inp.y.to(dev), 100, 4, 5.0, weights=inp.W.to(dev), mode="fp32")
    assert np.isfinite(float(loss))


def test_bf16_cfg5_full_size_vs_streamed_oracle():
    """BASELINE config 5, head part at full size: C = 85,742, D = 512, batch 2048, bf16."""
    dev = torch.device("cuda:0")
    B, D, Cn = 2048, 512, 85742
    inp = make_inputs(B, D, Cn)
    r = ref.asoftmax_head_streamed(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0, chunk=8192,
                                   dw_ranges=[(0, 4096), (40000, 44096), (Cn - 3000, Cn)], dtype=np.float32)
    loss, _, dX, dW = asoftmax_head(inp.X.to(dev), inp.y.to(dev), Cn, 4, 5.0, weights=inp.W.to(dev), mode="bf16",
                                    check_labels=True)
    torch.cuda.synchronize()
    assert abs(float(loss) - r.loss) <= 2e-3 * r.loss
    assert cosine(dX.cpu().numpy(), r.dX) >= 0.9999
    for (lo, hi), want in r.dW.items():
        got = dW[:, lo:hi].cpu().numpy()
        assert cosine(got, want) >= 0.9999, (lo, hi)
        assert np.abs(got - want).max() <= 2e-2 * np.abs(want).max(), (lo, hi)


def test_bf16_cfg4_shard_geometry_vs_streamed_oracle():
    """A config-4 shard at full size: batch 1024, D = 512, C_local = 125,000 (the 1/8 shard of
    C = 1,000,000), here as two such shards of a 250,000-class problem run one after the other
    through asm_forward_partial / asm_backward_partial and combined like the exchange would."""
    from tf_face_toolbox_b200.sharded import _CudaShard, shard_bounds
    dev = torch.device("cuda:0")
    B, D, Cn, G = 1024, 512, 250000, 2
    inp = make_inputs(B, D, Cn, seed=404)
    r = ref.asoftmax_head_streamed(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0, chunk=16384,
                                   dw_ranges=[(0, 8192), (125000, 125000 + 8192), (Cn - 4096, Cn)], dtype=np.float32)
    X, y = inp.X.to(dev), inp.y.to(dev)
    shards = []
    for g in range(G):
        lo, hi = shard_bounds(Cn, G, g)
        assert hi - lo == 125000
        shards.append((_CudaShard(D, Cn, lo, hi, 4, "bf16", g, G, dev), inp.W[:, lo:hi].contiguous().to(dev), lo, hi))
    stats_all = torch.stack([sh.forward_partial(X, y, Wg, 5.0) for sh, Wg, _, _ in shards]).contiguous()
    dX = torch.zeros(B, D, device=dev)
    dWs, losses = {}, []
    for sh, Wg, lo, hi in shards:
        loss, dXp, dWg = sh.backward_partial(stats_all, X, Wg)
        dX += dXp
        dWs[lo] = dWg
        losses.append(float(loss))
    torch.cuda.synchronize()
    assert losses[0] == losses[1] and abs(losses[0] - r.loss) <= 2e-3 * r.loss
    assert cosine(dX.cpu().numpy(), r.dX) >= 0.9999
    for (lo, hi), want in r.dW.items():
        base = 0 if lo < 125000 else 125000
        got = dWs[base][:, lo - base:hi - base].cpu().numpy()
        assert cosine(got, want) >= 0.9999, (lo, hi)
        assert np.abs(got - want).max() <= 2e-2 * np.abs(want).max(), (lo, hi)


def test_dw_rows_that_end_off_a_16_byte_boundary():
    """C % 4 == 2 (config 3's 85,742 is such a C): a dW row then starts AND ends 8 bytes off a
    16-byte boundary.  A TMA store box clipped at such an end was seen to clobber the first class
    of the next row (a lost update of the element next to the clip), which a cosine over the
    whole matrix does not notice: every element is checked here, on output buffers that hold
    NaN before the call."""
    dev = torch.device("cuda:0")
    B, D, Cn = 300, 192, 2002
    inp = make_inputs(B, D, Cn, seed=61)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    X, y, W = inp.X.to(dev), inp.y.to(dev), inp.W.to(dev)
    for _ in range(3):
        poison = torch.full((D, Cn), float("nan"), device=dev)
        del poison                                  # the caching allocator hands this block to dW next
        _, _, dX, dW = asoftmax_head(X, y, Cn, 4, 5.0, weights=W, mode="bf16")
        torch.cuda.synchronize()
        assert bool(torch.isfinite(dW).all()) and bool(torch.isfinite(dX).all())
        err = np.abs(dW.cpu().numpy() - r.dW).max(axis=0) / np.abs(r.dW).max()
        assert err.max() <= 2e-2, (int(err.argmax()), float(err.max()))


def test_bf16_embeddings_at_the_boundary():
    """asm_set_embedding_dtype: embeddings handed over as bf16 (bf16 mode) give the same result as the
    same values handed over as fp32 (the library would round them to bf16 itself)."""
    dev = torch.device("cuda:0")
    inp = make_inputs(300, 192, 2002, seed=61)
    X16 = inp.X.to(dev).to(torch.bfloat16)
    X32 = X16.float()
    y, W = inp.y.to(dev), inp.W.to(dev)
    la, _, dXa, dWa = asoftmax_head(X32, y, 2002, 4, 5.0, weights=W, mode="bf16")
    lb, _, dXb, dWb = asoftmax_head(X16, y, 2002, 4, 5.0, weights=W, mode="bf16")
    torch.cuda.synchronize()
    assert dXb.dtype == torch.float32
    # same operand bits; only the summation order inside the row norms differs (8 vs 4 elements per lane)
    assert float(la) == pytest.approx(float(lb), rel=1e-6)
    # (a 1e-7 relative change of n_i moves every exponent of the row; elements of dX that are a
    #  cancelling sum over the classes see it as an absolute error, so the bound is on max |diff| / max |dX|;
    #  handing over different VALUES, i.e. a second bf16 rounding, would show up at ~4e-3)
    ex = float((dXa - dXb).abs().max() / dXa.abs().max())
    ew = float((dWa - dWb).abs().max() / dWa.abs().max())
    assert ex <= 2e-5 and ew <= 2e-5, (ex, ew)
    r = ref.asoftmax_head(X32.cpu().numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    assert abs(float(lb) - r.loss) <= 2e-3 * r.loss and cosine(dXb.cpu().numpy(), r.dX) >= 0.9999
    with pytest.raises(TypeError):
        asoftmax_head(X16, y, 2002, 4, 5.0, weights=W, mode="fp32")
