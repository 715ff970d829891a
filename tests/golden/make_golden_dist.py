"""Golden vectors of the DATA-PARALLEL path from the UNMODIFIED reference: two gloo ranks on the CPU run
model.pretrain.InfoNCE (model/pretrain.py:98-190: shuffle-BN all-gather + rank-0 permutation broadcast, un-shuffle,
global enqueue) wrapped in DistributedDataParallel as main_nce.py:172 does, one training forward/backward each.
-> tests/golden/infonce_world2.npz (per-rank logits, replicated queue / pointer, DDP-averaged gradients).
Pins oracle.infonce_forward's simulated multi-rank world.  Needs a checkout of the reference:
    COCLR_REFERENCE=/path/to/CoCLR python tests/golden/make_golden_dist.py"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

CFG = dict(W=2, B=2, T=8, HW=64, K=32, ptr=8, threads=4, perm_seed=77)
GRAD_KEYS = ["encoder_q.0.Conv_1a.conv1.weight", "encoder_q.0.Conv_2c.bn1.weight", "encoder_q.0.Mixed_3c.branch1.1.conv2.weight",
             "encoder_q.0.Mixed_4d.branch2.0.conv.weight", "encoder_q.0.Mixed_5c.branch3.1.bn.bias", "encoder_q.4.weight"]


def rank_block(rank):
    g = torch.Generator().manual_seed(900 + rank)
    return torch.randn(CFG["B"], 2, 3, CFG["T"], CFG["HW"], CFG["HW"], generator=g)


def _worker(rank, port, out_dir):
    import torch.distributed as dist
    import make_golden as MG
    from oracle import coclr_oracle as O
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(CFG["threads"])
    torch.Tensor.cuda = lambda self, *a, **k: self          # pretrain.py:112,185 hard-code .cuda(); CPU shim
    dist.init_process_group("gloo", rank=rank, world_size=CFG["W"])
    ref = MG.import_reference()
    torch.manual_seed(0)
    model = ref.InfoNCE("s3d", 128, CFG["K"], 0.999, 0.07)
    sd = O.synth_state(O.infonce_shapes(128, CFG["K"]), seed=0, ptr=CFG["ptr"])
    model.load_state_dict(O.with_aliases(sd), strict=True)
    ddp = torch.nn.parallel.DistributedDataParallel(model)  # main_nce.py:172
    ddp.train()
    # only rank 0's permutation may matter (pretrain.py:112-115): the other rank draws from a different seed
    torch.manual_seed(CFG["perm_seed"] + 1000 * rank)
    logits, labels = ddp(rank_block(rank))
    loss = torch.nn.CrossEntropyLoss()(logits, labels)
    loss.backward()
    named = dict(model.named_parameters())
    res = {"logits": logits.detach().numpy(), "loss": np.float64(loss.item()), "queue": model.queue.numpy().copy(),
           "queue_ptr": model.queue_ptr.numpy().copy()}
    for k in GRAD_KEYS:
        res["grad/" + k] = named[k].grad.numpy().copy()
    res["ema/encoder_k.0.Conv_2c.conv1.weight"] = named["encoder_k.0.Conv_2c.conv1.weight"].detach().numpy().copy()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    dist.destroy_process_group()


def run_reference_world2(out_dir):
    import torch.multiprocessing as mp
    port = 29700 + (os.getpid() % 200)
    mp.spawn(_worker, args=(port, out_dir), nprocs=CFG["W"], join=True)
    r = [np.load(os.path.join(out_dir, "rank%d.npz" % i)) for i in range(CFG["W"])]
    out = {}
    for i in range(CFG["W"]):
        out["logits%d" % i] = r[i]["logits"]
        out["loss%d" % i] = r[i]["loss"]
    assert np.array_equal(r[0]["queue"], r[1]["queue"]) and np.array_equal(r[0]["queue_ptr"], r[1]["queue_ptr"])
    out["queue"], out["queue_ptr"] = r[0]["queue"], r[0]["queue_ptr"]
    for k in r[0].files:
        if k.startswith("grad/") or k.startswith("ema/"):
            assert np.array_equal(r[0][k], r[1][k]), k          # DDP leaves identical averaged gradients on every rank
            out[k] = r[0][k]
    return out


if __name__ == "__main__":
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        out = run_reference_world2(d)
    np.savez_compressed(os.path.join(HERE, "infonce_world2.npz"), **out)
    print("loss", out["loss0"], out["loss1"], "queue_ptr", out["queue_ptr"])
