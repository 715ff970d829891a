"""Pins the UberNCE / CoCLR restatements of the oracle against golden vectors from the unmodified reference
(tests/golden/{ubernce,coclr}_cfg1*.npz): at fp32 level under any thread count, and bit-for-bit with the reference's
thread count (8), which is how the golden vectors were made."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import coclr_oracle as O  # noqa: E402
import make_golden_ext as MX  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def oracle_ubernce():
    sh = O.infonce_shapes(128, MX.K)
    sh["queue_label"] = (MX.K,)
    sd = O.synth_state_ext(sh, seed=1, ptr=8)
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    b1, _, ids = MX.inputs(31)
    torch.manual_seed(78)
    idx = torch.randperm(MX.B)
    logits, mask = O.ubernce_forward(sd, b1, ids, idx)
    return sd, logits, mask


def oracle_coclr(full):
    sd = O.synth_state_ext(O.coclr_shapes(128, MX.K), seed=2, ptr=16, full=full)
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    b1, b2, ids = MX.inputs(32)
    torch.manual_seed(79)
    idx = torch.randperm(MX.B)
    logits, mask, is_full = O.coclr_forward(sd, b1, b2, ids, idx, queue_is_full=False, topk=5)
    return sd, logits, mask, is_full


def test_ubernce_oracle_matches_golden():
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    gold = np.load(os.path.join(G, "ubernce_cfg1.npz"))
    sd, logits, mask = oracle_ubernce()
    assert _rel(logits.detach().numpy(), gold["logits"]) < 2e-4
    assert np.array_equal(mask.numpy(), gold["mask"])
    assert mask.numpy()[:, 1:].any(), "the synthetic labels must produce positives in the queue"
    assert _rel(sd["queue"].numpy(), gold["queue"]) < 2e-4
    assert np.array_equal(sd["queue_label"].numpy(), gold["queue_label"])
    assert int(sd["queue_ptr"]) == int(gold["queue_ptr"][0]) == 12


@pytest.mark.parametrize("full", [True, False], ids=["topk", "warmup"])
def test_coclr_oracle_matches_golden(full):
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    gold = np.load(os.path.join(G, "coclr_cfg1.npz" if full else "coclr_cfg1_warmup.npz"))
    sd, logits, mask, is_full = oracle_coclr(full)
    assert _rel(logits.detach().numpy(), gold["logits"]) < 2e-4
    assert np.array_equal(mask.numpy(), gold["mask"])
    assert bool(gold["queue_is_full"]) == is_full == full
    if full:
        assert mask.numpy()[:, 1:].sum(1).min() >= 5      # top-5 mined positives per row
    assert _rel(sd["queue_second"].numpy(), gold["queue_second"]) < 2e-4
    assert np.array_equal(sd["queue_vname"].numpy(), gold["queue_vname"])
    assert np.array_equal(sd["queue_label"].numpy(), gold["queue_label"])


def test_ext_bitwise_vs_reference():
    torch.set_num_threads(8)
    ref_u = np.load(os.path.join(G, "ubernce_cfg1.npz"))
    _, logits, mask = oracle_ubernce()
    assert np.array_equal(logits.detach().numpy(), ref_u["logits"]) and np.array_equal(mask.numpy(), ref_u["mask"])
    ref_c = np.load(os.path.join(G, "coclr_cfg1.npz"))
    sd, logits, mask, _ = oracle_coclr(True)
    assert np.array_equal(logits.detach().numpy(), ref_c["logits"]) and np.array_equal(mask.numpy(), ref_c["mask"])
    assert np.array_equal(sd["queue_second"].numpy(), ref_c["queue_second"])
