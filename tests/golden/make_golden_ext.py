"""Golden vectors for UberNCE and CoCLR from the UNMODIFIED reference (model/pretrain.py:193-418) on CPU:
tests/golden/ubernce_cfg1.npz, tests/golden/coclr_cfg1.npz.  Needs a checkout of the reference:
    COCLR_REFERENCE=/path/to/CoCLR python tests/golden/make_golden_ext.py"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402
from oracle import coclr_oracle as O  # noqa: E402

K, B, T = 128, 4, 8


def inputs(seed):
    g = torch.Generator().manual_seed(seed)
    b1 = torch.randn(B, 2, 3, T, 128, 128, generator=g)
    b2 = torch.randn(B, 2, 3, T, 128, 128, generator=g)
    ids = torch.randint(0, 12, (B,), generator=g)
    return b1, b2, ids


def _init_pg():
    import torch.distributed as dist
    torch.set_num_threads(8)
    torch.Tensor.cuda = lambda self, *a, **k: self
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29582")
        dist.init_process_group("gloo", rank=0, world_size=1)


def run_ubernce():
    _init_pg()
    ref = MG.import_reference()
    torch.manual_seed(0)
    model = ref.UberNCE("s3d", 128, K, 0.999, 0.07)
    sh = O.infonce_shapes(128, K)
    sh["queue_label"] = (K,)
    sd = O.synth_state_ext(sh, seed=1, ptr=8)
    model.load_state_dict(O.with_aliases(sd), strict=True)
    model.train()
    b1, _, ids = inputs(31)
    torch.manual_seed(78)
    logits, mask = model(b1, ids)
    return {"logits": logits.detach().numpy(), "mask": mask.numpy(), "queue": model.queue.numpy().copy(),
            "queue_label": model.queue_label.numpy().copy(), "queue_ptr": model.queue_ptr.numpy().copy()}


def run_coclr(full=True, reverse=False):
    _init_pg()
    ref = MG.import_reference()
    torch.manual_seed(0)
    model = ref.CoCLR("s3d", 128, K, 0.999, 0.07, topk=5, reverse=reverse)
    sd = O.synth_state_ext(O.coclr_shapes(128, K), seed=2, ptr=16, full=full)
    model.load_state_dict(O.with_aliases(sd), strict=True)
    model.train()
    model.sampler.eval()
    b1, b2, ids = inputs(32)
    torch.manual_seed(79)
    logits, mask = model(b1, b2, ids)
    return {"logits": logits.detach().numpy(), "mask": mask.numpy(), "queue": model.queue.numpy().copy(),
            "queue_second": model.queue_second.numpy().copy(), "queue_vname": model.queue_vname.numpy().copy(),
            "queue_label": model.queue_label.numpy().copy(), "queue_ptr": model.queue_ptr.numpy().copy(),
            "queue_is_full": np.array(bool(model.queue_is_full))}


if __name__ == "__main__":
    np.savez_compressed(os.path.join(HERE, "ubernce_cfg1.npz"), **run_ubernce())
    np.savez_compressed(os.path.join(HERE, "coclr_cfg1.npz"), **run_coclr(True))
    np.savez_compressed(os.path.join(HERE, "coclr_cfg1_warmup.npz"), **run_coclr(False))
    print("written")
