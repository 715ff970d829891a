"""Golden data for the drop-in checks of the training scripts (tests/test_host_cpu.py), taken from the UNMODIFIED
reference's main_nce.py / main_coclr.py.  Those scripts cannot be imported (tensorboardX / lmdb are absent), so their
source text is parsed or executed piecewise:
  * reference_cli.json: every command-line option of both scripts (whether it takes a value, whether nargs=2);
  * reference_two_checkpoint.npz: the key mapping of main_coclr.py's two-checkpoint initialisation (--pretrain A B,
    main_coclr.py:250-302) run on checkpoints whose values name their own keys;
  * reference_losses.npz: multi_nce_loss (main_coclr.py:343-346) and the UberNCE loss line (main_nce.py:321-322) on
    three seeded (logits, mask) draws.
Needs a checkout of the reference:  COCLR_REFERENCE=/path/to/CoCLR python tests/golden/make_golden_cli.py"""
import ast
import json
import os
import re
import sys
import textwrap
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("COCLR_REFERENCE", "")


def ref_flags(path):
    out = {}
    for m in re.finditer(r"add_argument\(([^)]*)\)", open(path).read()):
        names = re.findall(r"'(-{1,2}[\w-]+)'", m.group(1))
        for n in names:
            out[n] = ["store_true" not in m.group(1), "nargs=2" in m.group(1)]
    return out


def checkpoint_keys():
    """state_dict keys of the two checkpoints of the merge: a CoCLR one (has sampler.* and queue_second) and an
    InfoNCE one, as this repository's modules (whose keys equal the reference's) write them."""
    from model.pretrain import CoCLR, InfoNCE
    return list(CoCLR("s3d", 128, 128, topk=5).state_dict()), list(InfoNCE("s3d", 128, 128).state_dict())


def two_checkpoint_merge(first_keys, second_keys):
    """Runs the reference's merge block on two checkpoints whose values name their origin ('first:<key>')."""
    lines = open(os.path.join(REF, "main_coclr.py")).read().splitlines()
    start = next(i for i, ln in enumerate(lines) if ln.strip().startswith("elif args.pretrain != ['random', 'random']"))
    end = next(i for i in range(start, len(lines)) if lines[i].strip().startswith("neq_load_customized("))
    block = textwrap.dedent("\n".join(lines[start:end])).replace("elif ", "if ", 1)
    ckpts = {"A": {"epoch": 7, "state_dict": {k: "first:" + k for k in first_keys}},
             "B": {"epoch": 9, "state_dict": {k: "second:" + k for k in second_keys}}}
    fake_torch = types.SimpleNamespace(load=lambda p, map_location=None: ckpts[p], device=torch.device)
    fake_os = types.SimpleNamespace(path=types.SimpleNamespace(isfile=lambda p: p in ckpts))
    ns = {"args": types.SimpleNamespace(pretrain=["A", "B"]), "torch": fake_torch, "os": fake_os, "print": lambda *a: None}
    exec(compile(block, "reference_two_checkpoint_merge", "exec"), ns)
    return ns["state_dict"]


def loss_draws():
    lines = open(os.path.join(REF, "main_coclr.py")).read()
    fn = [n for n in ast.parse(lines).body if isinstance(n, ast.FunctionDef) and n.name == "multi_nce_loss"][0]
    ns = {"torch": torch, "F": F}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "ref_multi_nce_loss", "exec"), ns)
    uber = [ln.strip() for ln in open(os.path.join(REF, "main_nce.py")).read().splitlines()
            if ln.strip().startswith("loss = - (F.log_softmax(output, dim=1) * target)")]
    assert len(uber) == 1
    g = torch.Generator().manual_seed(9)
    out = {k: [] for k in ("logits", "mask", "multi_nce_loss", "ubernce_loss")}
    for _ in range(3):
        logits = torch.randn(6, 1 + 40, generator=g) * 4
        mask = torch.rand(6, 41, generator=g) < 0.15
        mask[:, 0] = True
        env = {"F": F, "output": logits, "target": mask}
        exec(uber[0], env)
        out["logits"].append(logits.numpy())
        out["mask"].append(mask.numpy())
        out["multi_nce_loss"].append(ns["multi_nce_loss"](logits, mask).numpy())
        out["ubernce_loss"].append(env["loss"].mean().numpy())
    return {k: np.stack(v) for k, v in out.items()}


if __name__ == "__main__":
    if not os.path.isfile(os.path.join(REF, "main_coclr.py")):
        raise SystemExit("set COCLR_REFERENCE to a checkout of the reference (TengdaHan/CoCLR)")
    first, second = checkpoint_keys()
    cli = {"main_nce": ref_flags(os.path.join(REF, "main_nce.py")),
           "main_coclr": ref_flags(os.path.join(REF, "main_coclr.py"))}
    with open(os.path.join(HERE, "reference_cli.json"), "w") as fh:
        json.dump(cli, fh, indent=0, sort_keys=True)
    merged = two_checkpoint_merge(first, second)
    np.savez_compressed(os.path.join(HERE, "reference_two_checkpoint.npz"), first_keys=np.array(first),
                        second_keys=np.array(second), merged_keys=np.array(list(merged)),
                        merged_values=np.array(list(merged.values())))
    np.savez_compressed(os.path.join(HERE, "reference_losses.npz"), **loss_draws())
    print("written")
