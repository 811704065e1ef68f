"""Whole-model checks on the GPU: our kernels vs the PyTorch oracle of the same ops, eager vs CUDA graph."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu

import tiny_deepspeed_b200 as tds  # noqa: E402
from tiny_deepspeed_b200 import ops  # noqa: E402
from tiny_deepspeed_b200.models.gpt2 import GPT2Model, gpt2_config  # noqa: E402


def _mk(seed=0, **kw):
    torch.manual_seed(seed)
    cfg = gpt2_config("tiny", n_layer=2, n_head=4, n_embd=256, vocab_size=2048, block_size=256, **kw)
    return cfg, GPT2Model(cfg).to(device="cuda", dtype=torch.bfloat16)


def test_model_grads_match_oracle():
    cfg, m = _mk()
    x = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    y = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    _, loss = m(x, y)
    loss.backward()
    got = {n: p.grad.float().clone() for n, p in m.named_parameters()}
    for p in m.parameters():
        p.grad = None
    ops.force_torch(True)
    try:
        _, rloss = m(x, y)
        rloss.backward()
    finally:
        ops.force_torch(False)
    torch.testing.assert_close(loss, rloss, rtol=2e-3, atol=2e-3)
    for n, p in m.named_parameters():
        ref = p.grad.float()
        rel = (got[n] - ref).norm() / (ref.norm() + 1e-12)
        assert rel < 3e-2, (n, float(rel))


def test_training_decreases_loss_and_graph_matches_eager():
    cfg, m1 = _mk(1)
    m2 = copy.deepcopy(m1)
    x = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    y = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    o1 = tds.AdamW(m1.named_parameters(), lr=1e-3, weight_decay=0.1)
    o2 = tds.AdamW(m2.named_parameters(), lr=1e-3, weight_decay=0.1)
    s1 = tds.TrainStep(m1, o1, use_graph=False)
    s2 = tds.TrainStep(m2, o2, use_graph=True, warmup=2)
    l1 = [float(s1(x, y)) for _ in range(8)]
    l2 = [float(s2(x, y)) for _ in range(8)]
    assert s2.graph is not None and s2.launches_per_step > 20
    assert l1[-1] < l1[0] - 0.05
    assert l2 == pytest.approx(l1, rel=2e-3, abs=2e-3), (l1, l2)
    for (n, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        torch.testing.assert_close(a.float(), b.float(), rtol=1e-2, atol=1e-3, msg=n)


def test_smoke_entry():
    import __graft_entry__ as g
    g.smoke()


def test_bench_dump_outputs_reproducible(tmp_path):
    """bench.py --dump-outputs end to end (tiny model): the JSON line reports the requested steps, loss.npy is the reported
    final loss, and a second run with the same arguments dumps the same arrays (up to atomics-order rounding)."""
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    from dist_utils import free_port

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = []
    for tag in ("a", "b"):
        out = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--model", "tiny", "--modes", "none", "--steps", "3",
                            "--warmup", "2", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600,
                           env={**os.environ, "MASTER_PORT": str(free_port())})
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 3
        loss = np.load(out / "loss.npy")
        assert loss.dtype == np.float32 and loss.tolist() == [pytest.approx(line["final_loss"], rel=1e-6)]
        runs.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = runs
    assert set(a) == set(b) and any(k.startswith("master.") for k in a) and sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all(), k
        np.testing.assert_allclose(a[k], b[k], rtol=1e-3, atol=1e-3, err_msg=k)


def test_optimizer_in_backward_overlap_matches_plain_step():
    cfg, m1 = _mk(2)
    m2 = copy.deepcopy(m1)
    x = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    y = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    o1 = tds.AdamW(m1.named_parameters(), lr=1e-3, weight_decay=0.1)
    o2 = tds.AdamW(m2.named_parameters(), lr=1e-3, weight_decay=0.1)
    s1 = tds.TrainStep(m1, o1, use_graph=False, overlap_step=False)
    s2 = tds.TrainStep(m2, o2, use_graph=False, overlap_step=True)
    s2.overlap.bucket_bytes = 64 << 10          # several buckets even for the tiny model
    l1 = [float(s1(x, y)) for _ in range(6)]
    l2 = [float(s2(x, y)) for _ in range(6)]
    assert s2.overlap.stats["overlapped_buckets"] > 0
    assert o1.step_count == o2.step_count == 6
    assert l2 == pytest.approx(l1, rel=1e-4, abs=1e-4), (l1, l2)
    for (n, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        torch.testing.assert_close(a.float(), b.float(), rtol=1e-3, atol=1e-4, msg=n)


def _fp32_oracle_check(m, x, y):
    _, loss = m(x, y)
    loss.backward()
    got = {n: p.grad.clone() for n, p in m.named_parameters()}
    assert all(g.dtype == torch.float32 for g in got.values())
    for p in m.parameters():
        p.grad = None
    ops.force_torch(True)
    try:
        _, rloss = m(x, y)
        rloss.backward()
    finally:
        ops.force_torch(False)
    torch.testing.assert_close(loss, rloss, rtol=1e-3, atol=1e-3)
    for n, p in m.named_parameters():
        rel = (got[n] - p.grad).norm() / (p.grad.norm() + 1e-12)
        assert rel < 2e-2, (n, float(rel))
        p.grad = None


def test_fp32_model_matches_oracle_and_trains():
    """fp32 parameters (the reference's dtype, example/single_device/train.py:16): GEMMs run as TF32 on tcgen05, LN / CE /
    Adam in fp32, the attention core on the bf16 flash kernels."""
    import gc
    torch.manual_seed(3)
    cfg = gpt2_config("tiny", n_layer=2, n_head=4, n_embd=256, vocab_size=2048, block_size=256, bias=True)
    m = GPT2Model(cfg).to(device="cuda", dtype=torch.float32)
    x = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    y = torch.randint(0, cfg.vocab_size, (2, 256), device="cuda")
    # in a helper so every eager autograd graph (logits, losses) is gone afterwards: their AccumulateGrad nodes are bound
    # to the default stream and must not be reused inside the capture (torch's usual rule for CUDA-graph capture)
    _fp32_oracle_check(m, x, y)
    gc.collect()
    opt = tds.AdamW(m.named_parameters(), lr=1e-3, weight_decay=0.1)
    step = tds.TrainStep(m, opt, use_graph=True, warmup=2)
    losses = [float(step(x, y)) for _ in range(8)]
    assert losses[-1] < losses[0] - 0.05, losses
