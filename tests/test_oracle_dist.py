"""Pins the oracle's SIMULATED multi-rank world (oracle.infonce_forward with several blocks: shuffle-BN permutation,
un-shuffle, global enqueue; model/pretrain.py:82-143) and the DDP gradient averaging (main_nce.py:172) against the
unmodified reference run as two real gloo ranks (tests/golden/infonce_world2.npz): (1) at fp32 level under any thread
count; (2) bit-for-bit with the thread count the golden vectors were made with (make_golden_dist.CFG)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import coclr_oracle as O  # noqa: E402
import make_golden_dist as MD  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "infonce_world2.npz")


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _oracle_world2():
    c = MD.CFG
    torch.set_num_threads(c["threads"])
    sd = O.synth_state(O.infonce_shapes(128, c["K"]), seed=0, ptr=c["ptr"])
    qkeys = O.param_keys(sd, "encoder_q.")
    for k in qkeys:
        sd[k].requires_grad_(True)
    blocks = [MD.rank_block(r) for r in range(c["W"])]
    torch.manual_seed(c["perm_seed"])                       # rank 0's draw (pretrain.py:112)
    idx = torch.randperm(c["B"] * c["W"])
    logits, labels = O.infonce_forward(sd, blocks, idx)
    losses = [O.infonce_loss(lg, labels) for lg in logits]
    (sum(losses) / c["W"]).backward()                       # DDP: mean of the per-rank gradients
    return sd, logits, losses


def _check(sd, logits, losses, gold, tol_fwd, tol_grad):
    c = MD.CFG
    for r in range(c["W"]):
        assert logits[r].shape == (c["B"], 1 + c["K"])
        assert _rel(logits[r].detach().numpy(), gold["logits%d" % r]) <= tol_fwd, r
        assert abs(float(losses[r]) - float(gold["loss%d" % r])) <= max(tol_fwd, 1e-12) * max(1.0, abs(float(gold["loss%d" % r])))
    assert _rel(sd["queue"].numpy(), gold["queue"]) <= tol_fwd
    assert int(sd["queue_ptr"]) == int(gold["queue_ptr"][0]) == c["ptr"] + c["B"] * c["W"]
    assert _rel(sd["encoder_k.0.Conv_2c.conv1.weight"].detach().numpy(), gold["ema/encoder_k.0.Conv_2c.conv1.weight"]) <= 1e-6
    for k in MD.GRAD_KEYS:
        assert _rel(sd[k].grad.numpy(), gold["grad/" + k]) <= tol_grad, k


def test_oracle_world2_matches_golden():
    sd, logits, losses = _oracle_world2()
    # thread counts / reduction order may differ from the generating run: fp32-level forward, loose gradient bound
    _check(sd, logits, losses, np.load(GOLD), tol_fwd=2e-4, tol_grad=5e-2)


def test_oracle_world2_bitwise_vs_reference():
    out = np.load(GOLD)
    sd, logits, losses = _oracle_world2()
    for r in range(MD.CFG["W"]):
        assert np.array_equal(logits[r].detach().numpy(), out["logits%d" % r]), "per-rank logits differ from the reference"
    assert np.array_equal(sd["queue"].numpy(), out["queue"])
    _check(sd, logits, losses, out, tol_fwd=0.0, tol_grad=1e-5)
