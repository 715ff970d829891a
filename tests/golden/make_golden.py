"""Generates tests/golden/infonce_cfg1.npz (and, with the argument `r50` / `s3dg`, infonce_r50.npz / infonce_s3dg.npz) by running the UNMODIFIED reference (TengdaHan/CoCLR,
model/pretrain.py InfoNCE) on BASELINE.json config 1 (S3D, moco-k=128, bs=4,
seq_len=8, 128x128, CPU) from the deterministic synthetic state of oracle.coclr_oracle.synth_state.

Needs a checkout of the reference, named by the environment variable COCLR_REFERENCE:
    COCLR_REFERENCE=/path/to/CoCLR python tests/golden/make_golden.py [r50|s3dg]
The .npz stores reference outputs (logits, loss, updated queue/ptr, selected gradients and
post-EMA key weights); inputs are regenerated from seeds by the tests.  The companion <name>_state.npz holds a
sample of every entry of the reference model's state_dict after the step (see state_sample).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("COCLR_REFERENCE", "")


def make_inputs(B=4, T=8, HW=128, seed=1234):  # noqa
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 2, 3, T, HW, HW, generator=g)


def make_inputs_shifted(B=4, T=8, HW=64, seed=1234):  # noqa
    """Noise clips plus a per-clip colour offset and a per-clip spatial ramp, so that clips stay distinguishable after
    the global average pool (pure noise gives q == k for every pair and a saturated loss)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 2, 3, T, HW, HW, generator=g)
    x = x + 1.5 * torch.randn(B, 2, 3, 1, 1, 1, generator=g)
    ramp = torch.linspace(-1, 1, HW).view(1, 1, 1, 1, 1, HW)
    return x + torch.randn(B, 2, 3, 1, 1, 1, generator=g) * ramp


def compact(a, limit=16384):
    """Large arrays are stored as a strided sample (every n-th element of the flattened array) + their L2 norm."""
    a = np.asarray(a)
    if a.size <= limit:
        return a.copy(), None
    stride = -(-a.size // limit)
    return a.reshape(-1)[::stride].copy(), np.float64(np.linalg.norm(a.astype(np.float64)))


GRAD_KEYS = ["encoder_q.0.Conv_1a.conv1.weight", "encoder_q.0.Conv_1a.bn2.weight", "encoder_q.0.Conv_2c.conv2.weight",
             "encoder_q.0.Mixed_3b.branch2.1.conv1.weight", "encoder_q.0.Mixed_4c.branch2.0.conv.weight",
             "encoder_q.0.Mixed_4f.branch3.1.bn.bias", "encoder_q.0.Mixed_5c.branch1.1.conv2.weight",
             "encoder_q.2.weight", "encoder_q.4.bias"]


def import_reference():
    """Import the UNMODIFIED reference's model.pretrain without clashing with this repo's own `model` /
    `backbone` packages (same top-level names by design: they are drop-ins)."""
    import importlib
    if not os.path.isdir(os.path.join(REF, "model")):
        raise SystemExit("set COCLR_REFERENCE to a checkout of the reference (TengdaHan/CoCLR)")
    clash = lambda k: k in ("model", "backbone") or k.startswith("model.") or k.startswith("backbone.")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if clash(k)}
    sys.path.insert(0, REF)
    try:
        mod = importlib.import_module("model.pretrain")
        assert mod.__file__.startswith(REF), mod.__file__
    finally:
        sys.path.remove(REF)
        for k in list(sys.modules):
            if clash(k):
                sys.modules.pop(k)
        sys.modules.update(saved)
    return mod


def state_sample(sd, limit=128):
    """Strided sample (compact) of every entry of a state_dict, packed as three arrays: the keys, the end offset of
    each key's sample and all samples back to back as float32.  The post-step state of the reference is compared on
    it; one array per key would cost more in archive headers than in data."""
    keys = sorted(sd)
    parts = [compact(sd[k].detach().float().numpy(), limit)[0].reshape(-1) for k in keys]
    return {"state_keys": np.array(keys), "state_ends": np.cumsum([p.size for p in parts]),
            "state_values": np.concatenate(parts).astype(np.float32)}


GRAD_KEYS_R50 = ["encoder_q.0.conv1.weight", "encoder_q.0.bn1.weight", "encoder_q.0.layer1.0.conv2.weight",
                 "encoder_q.0.layer1.0.downsample.0.weight", "encoder_q.0.layer1.0.downsample.1.bias",
                 "encoder_q.0.layer2.3.conv3.weight", "encoder_q.0.layer3.0.conv1.weight", "encoder_q.0.layer3.5.bn3.weight",
                 "encoder_q.0.layer4.2.conv1.weight", "encoder_q.2.weight", "encoder_q.4.bias"]
R50_CFG = dict(K=128, B=4, T=8, HW=64, ptr=16)     # BASELINE.json config 5 (--net r50) at a CPU-sized shape


# S3D-G (`--net s3dg`, select_backbone.py:8-9: S3D with a SelfGating on every SepInception branch output)
GRAD_KEYS_S3DG = ["encoder_q.0.Conv_1a.conv1.weight", "encoder_q.0.Conv_2c.conv2.weight",
                  "encoder_q.0.Mixed_3b.gating_b1.fc.weight", "encoder_q.0.Mixed_3b.gating_b1.fc.bias",
                  "encoder_q.0.Mixed_3c.branch1.1.conv1.weight", "encoder_q.0.Mixed_4c.gating_b0.fc.weight",
                  "encoder_q.0.Mixed_4f.branch3.1.bn.bias", "encoder_q.0.Mixed_5c.gating_b3.fc.bias",
                  "encoder_q.0.Mixed_5c.branch1.1.conv2.weight", "encoder_q.2.weight", "encoder_q.4.bias"]
S3DG_CFG = dict(K=128, B=4, T=8, HW=128, ptr=16)     # config 1 shape (the 64x64 r50 shape leaves Mixed_5 BatchNorms 16 samples)


def run_reference(K=128, B=4, T=8, ptr=16, threads=8, network="s3d", HW=128):
    import torch.distributed as dist
    InfoNCE = import_reference().InfoNCE  # the unmodified reference
    from oracle import coclr_oracle as O
    torch.set_num_threads(threads)
    torch.Tensor.cuda = lambda self, *a, **k: self  # pretrain.py:112,185 hard-code .cuda(); CPU shim
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29581")
        dist.init_process_group("gloo", rank=0, world_size=1)
    torch.manual_seed(0)
    model = InfoNCE(network, 128, K, 0.999, 0.07)
    sd = O.synth_state(O.infonce_shapes(128, K, network=network), seed=0, ptr=ptr)
    model.load_state_dict(O.with_aliases(sd), strict=True)
    model.train()
    block = make_inputs(B, T, HW) if network == "s3d" else make_inputs_shifted(B, T, HW)
    torch.manual_seed(77)  # fixes the torch.randperm draw of _batch_shuffle_ddp (pretrain.py:112)
    logits, labels = model(block)
    loss = torch.nn.CrossEntropyLoss()(logits, labels)
    loss.backward()
    out = {"logits": logits.detach().numpy(), "loss": np.float64(loss.item()),
           "queue": model.queue.numpy().copy(), "queue_ptr": model.queue_ptr.numpy().copy()}
    named = dict(model.named_parameters())
    if network == "s3d":
        for k in GRAD_KEYS:
            out["grad/" + k] = named[k].grad.numpy().copy()
    if network == "s3dg":
        for k in GRAD_KEYS_S3DG:
            out["grad/" + k], nrm = compact(named[k].grad.numpy())
            if nrm is not None:
                out["gradnorm/" + k] = nrm
        out["ema/encoder_k.0.Mixed_4b.gating_b2.fc.weight"] = named["encoder_k.0.Mixed_4b.gating_b2.fc.weight"].detach().numpy().copy()
    if network == "r50":
        for k in GRAD_KEYS_R50:
            out["grad/" + k], nrm = compact(named[k].grad.numpy())
            if nrm is not None:
                out["gradnorm/" + k] = nrm
        full = model.state_dict()
        out["ema/encoder_k.0.layer2.0.conv2.weight"] = named["encoder_k.0.layer2.0.conv2.weight"].detach().numpy().copy()
        out["bn/encoder_q.0.layer1.0.downsample.1.running_mean"] = full["encoder_q.0.layer1.0.downsample.1.running_mean"].numpy().copy()
        out["bn/encoder_k.0.layer4.2.bn3.running_var"] = full["encoder_k.0.layer4.2.bn3.running_var"].numpy().copy()
        return out, model
    out["ema/encoder_k.0.Conv_2c.conv1.weight"] = named["encoder_k.0.Conv_2c.conv1.weight"].detach().numpy().copy()
    out["bn/encoder_q.0.Conv_1a.bn1.running_mean"] = model.state_dict()["encoder_q.0.Conv_1a.bn1.running_mean"].numpy().copy()
    out["bn/encoder_k.0.Mixed_5c.branch0.0.bn.running_var"] = model.state_dict()["encoder_k.0.Mixed_5c.branch0.0.bn.running_var"].numpy().copy()
    return out, model


if __name__ == "__main__":
    if "s3dg" in sys.argv[1:]:
        name, (out, model) = "infonce_s3dg", run_reference(network="s3dg", **S3DG_CFG)
    elif "r50" in sys.argv[1:]:
        name, (out, model) = "infonce_r50", run_reference(network="r50", **R50_CFG)
    else:
        name, (out, model) = "infonce_cfg1", run_reference()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    np.savez_compressed(os.path.join(HERE, name + "_state.npz"), **state_sample(model.state_dict()))
    print("loss", out["loss"], "logits[0,:4]", out["logits"][0, :4])
