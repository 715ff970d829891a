"""Pins the oracle (oracle/coclr_oracle.py) against the golden vectors generated from the unmodified reference
(tests/golden/infonce_cfg1.npz, BASELINE.json config 1, and the r50 / s3dg files): (1) at fp32 level under any thread
count; (2) bit-for-bit with the reference's thread count (8), which is how the golden vectors were made, on the outputs,
the stored gradients and a sample of every entry of the reference's post-step state_dict (tests/golden/*_state.npz)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import coclr_oracle as O  # noqa: E402
import make_golden as MG  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "infonce_cfg1.npz")


def _oracle_step(K=128, B=4, T=8, ptr=16):
    sd = O.synth_state(O.infonce_shapes(128, K), seed=0, ptr=ptr)
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    block = MG.make_inputs(B, T)
    torch.manual_seed(77)
    idx = torch.randperm(B)
    logits, labels = O.infonce_forward(sd, [block], idx)
    loss = O.infonce_loss(logits[0], labels)
    loss.backward()
    return sd, logits[0], loss


def _rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _check_state(sd, name):
    """Every post-step buffer / weight of the oracle against the sample of the reference's state_dict (make_golden.state_sample)."""
    st = np.load(os.path.join(ROOT, "tests", "golden", name + "_state.npz"))
    ends = st["state_ends"]
    ref = {str(k): st["state_values"][(ends[i - 1] if i else 0):ends[i]] for i, k in enumerate(st["state_keys"])}
    assert set(ref) == set(O.with_aliases(sd))
    for k, v in sd.items():
        assert _rel(MG.compact(v.detach().float().numpy(), 128)[0].reshape(-1), ref[k]) < 1e-6, k


def test_oracle_matches_golden():
    gold = np.load(GOLD)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    sd, logits, loss = _oracle_step()
    assert _rel(logits.detach().numpy(), gold["logits"]) < 2e-4
    assert abs(loss.item() - float(gold["loss"])) < 2e-4 * max(1.0, abs(float(gold["loss"])))
    assert _rel(sd["queue"].numpy(), gold["queue"]) < 2e-4
    assert int(sd["queue_ptr"]) == int(gold["queue_ptr"][0]) == 20
    # EMA and BN buffers are elementwise / reductions: tight
    assert _rel(sd["encoder_k.0.Conv_2c.conv1.weight"].detach().numpy(),
                gold["ema/encoder_k.0.Conv_2c.conv1.weight"]) < 1e-6
    assert _rel(sd["encoder_q.0.Conv_1a.bn1.running_mean"].numpy(),
                gold["bn/encoder_q.0.Conv_1a.bn1.running_mean"]) < 1e-5
    assert _rel(sd["encoder_k.0.Mixed_5c.branch0.0.bn.running_var"].numpy(),
                gold["bn/encoder_k.0.Mixed_5c.branch0.0.bn.running_var"]) < 1e-4
    # gradients: the reference disagrees with itself by ~1e-2 under summation-order changes
    # (SURVEY.md section 7), so only a loose bound is meaningful across thread counts
    for k in MG.GRAD_KEYS:
        assert _rel(sd[k].grad.numpy(), gold["grad/" + k]) < 5e-2, k


def test_oracle_bitwise_vs_reference():
    torch.set_num_threads(8)
    out = np.load(GOLD)
    sd, logits, loss = _oracle_step()
    assert np.array_equal(logits.detach().numpy(), out["logits"])
    assert loss.item() == float(out["loss"])
    assert np.array_equal(sd["queue"].numpy(), out["queue"])
    for k in MG.GRAD_KEYS:
        assert _rel(sd[k].grad.numpy(), out["grad/" + k]) < 1e-6, k
    # every post-step buffer / key-encoder weight
    _check_state(sd, "infonce_cfg1")


def test_alias_expansion_covers_reference_keys():
    sd = O.synth_state(O.infonce_shapes(128, 128))
    full = O.with_aliases(sd)
    assert "encoder_q.0.block1.0.conv1.weight" in full
    assert full["encoder_k.0.block5.2.branch3.1.bn.bias"] is sd["encoder_k.0.Mixed_5c.branch3.1.bn.bias"]
    # 235 parameter tensors per encoder, as the reference's named_parameters() reports (SURVEY.md K12)
    assert len(O.param_keys(sd, "encoder_q.")) == 235


# ---- r50 (ResNet2d3d-50, BASELINE.json config 5) -------------------------------------------------
GOLD_R50 = os.path.join(ROOT, "tests", "golden", "infonce_r50.npz")


def _oracle_step_r50():
    c = MG.R50_CFG
    sd = O.synth_state(O.infonce_shapes(128, c["K"], network="r50"), seed=0, ptr=c["ptr"])
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    block = MG.make_inputs_shifted(c["B"], c["T"], c["HW"])
    torch.manual_seed(77)
    idx = torch.randperm(c["B"])
    logits, labels = O.infonce_forward(sd, [block], idx)
    loss = O.infonce_loss(logits[0], labels)
    loss.backward()
    return sd, logits[0], loss


def test_oracle_r50_matches_golden():
    gold = np.load(GOLD_R50)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    sd, logits, loss = _oracle_step_r50()
    assert logits.shape == (4, 129)
    assert _rel(logits.detach().numpy(), gold["logits"]) < 2e-4
    assert _rel(sd["queue"].numpy(), gold["queue"]) < 2e-4
    assert int(sd["queue_ptr"]) == int(gold["queue_ptr"][0]) == 20
    assert _rel(sd["encoder_k.0.layer2.0.conv2.weight"].detach().numpy(), gold["ema/encoder_k.0.layer2.0.conv2.weight"]) < 1e-6
    assert _rel(sd["encoder_q.0.layer1.0.downsample.1.running_mean"].numpy(),
                gold["bn/encoder_q.0.layer1.0.downsample.1.running_mean"]) < 1e-5
    assert _rel(sd["encoder_k.0.layer4.2.bn3.running_var"].numpy(), gold["bn/encoder_k.0.layer4.2.bn3.running_var"]) < 1e-4
    for k in MG.GRAD_KEYS_R50:
        got, _ = MG.compact(sd[k].grad.numpy())
        assert _rel(got, gold["grad/" + k]) < 5e-2, k


def test_r50_inventory():
    sh = O.r50_shapes("")
    convs = [k for k, v in sh.items() if len(v) == 5]
    assert len(convs) == 53                                            # SURVEY.md row a14
    n_params = sum(int(np.prod(v)) for k, v in sh.items() if k.endswith(".weight") or k.endswith(".bias"))
    assert n_params == 31_632_960 or abs(n_params - 31.7e6) < 0.2e6, n_params


def _check_grads(sd, out, keys):
    """Gradients stored whole, or as a strided sample plus the L2 norm of the whole tensor (make_golden.compact)."""
    for k in keys:
        got, nrm = MG.compact(sd[k].grad.numpy())
        assert _rel(got, out["grad/" + k]) < 1e-6, k
        if nrm is not None:
            assert abs(nrm - float(out["gradnorm/" + k])) < 1e-6 * float(out["gradnorm/" + k]), k


def test_oracle_r50_bitwise_vs_reference():
    torch.set_num_threads(8)
    out = np.load(GOLD_R50)
    sd, logits, loss = _oracle_step_r50()
    assert np.array_equal(logits.detach().numpy(), out["logits"])
    assert loss.item() == float(out["loss"])
    assert np.array_equal(sd["queue"].numpy(), out["queue"])
    _check_grads(sd, out, MG.GRAD_KEYS_R50)
    _check_state(sd, "infonce_r50")


def test_oracle_adam_is_torch_optim_adam():
    """oracle.adam_step restates torch.optim.Adam(params, lr, weight_decay) as the reference builds it
    (main_nce.py:190-200: one group, lr 1e-3, wd 1e-5, coupled L2): several steps on random tensors, bit-for-bit."""
    g = torch.Generator().manual_seed(4)
    shapes = [(64, 3, 1, 7, 7), (192,), (128, 1024, 1, 1, 1), (17,)]
    ps = [torch.randn(s, generator=g) * 0.1 for s in shapes]
    ref_params = [torch.nn.Parameter(p.clone()) for p in ps]
    opt = torch.optim.Adam([{"params": ref_params}], lr=1e-3, weight_decay=1e-5)
    mine = {str(i): p.clone() for i, p in enumerate(ps)}
    state = {}
    for step in range(5):
        grads = [torch.randn(s, generator=g) * (0.01 + 0.1 * step) for s in shapes]
        for p, gr in zip(ref_params, grads):
            p.grad = gr.clone()
        opt.step()
        O.adam_step(mine, {str(i): gr for i, gr in enumerate(grads)}, state, lr=1e-3, weight_decay=1e-5)
        for i, p in enumerate(ref_params):
            assert torch.equal(mine[str(i)], p.detach()), (step, i)


# ---- s3dg (S3D with feature gating, `--net s3dg`; backbone/s3dg.py:68-78,107-112,125-129) ---------
GOLD_S3DG = os.path.join(ROOT, "tests", "golden", "infonce_s3dg.npz")


def _oracle_step_s3dg():
    c = MG.S3DG_CFG
    sd = O.synth_state(O.infonce_shapes(128, c["K"], network="s3dg"), seed=0, ptr=c["ptr"])
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    block = MG.make_inputs_shifted(c["B"], c["T"], c["HW"])
    torch.manual_seed(77)
    idx = torch.randperm(c["B"])
    logits, labels = O.infonce_forward(sd, [block], idx)
    loss = O.infonce_loss(logits[0], labels)
    loss.backward()
    return sd, logits[0], loss


def test_oracle_s3dg_matches_golden():
    gold = np.load(GOLD_S3DG)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    sd, logits, loss = _oracle_step_s3dg()
    assert logits.shape == (4, 129)
    assert _rel(logits.detach().numpy(), gold["logits"]) < 2e-4
    assert _rel(sd["queue"].numpy(), gold["queue"]) < 2e-4
    assert int(sd["queue_ptr"]) == int(gold["queue_ptr"][0]) == 20
    assert _rel(sd["encoder_k.0.Mixed_4b.gating_b2.fc.weight"].detach().numpy(),
                gold["ema/encoder_k.0.Mixed_4b.gating_b2.fc.weight"]) < 1e-6
    for k in MG.GRAD_KEYS_S3DG:
        got, _ = MG.compact(sd[k].grad.numpy())
        assert _rel(got, gold["grad/" + k]) < 5e-2, k
    # 9 SepInception blocks x 4 SelfGating x (weight, bias) on top of S3D's 235 tensors
    assert len(O.param_keys(sd, "encoder_q.")) == 235 + 72


def test_oracle_s3dg_bitwise_vs_reference():
    torch.set_num_threads(8)
    out = np.load(GOLD_S3DG)
    sd, logits, loss = _oracle_step_s3dg()
    assert np.array_equal(logits.detach().numpy(), out["logits"])
    assert loss.item() == float(out["loss"])
    assert np.array_equal(sd["queue"].numpy(), out["queue"])
    _check_grads(sd, out, MG.GRAD_KEYS_S3DG)
    _check_state(sd, "infonce_s3dg")
