#!/usr/bin/env python
"""Benchmark of the CoCLR hot path (BASELINE.json metric: clips/sec, S3D InfoNCE, 32 x 128^2 clips, K=2048).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

A "step" is one full training step on a per-GPU batch of 32 clip pairs: q-encoder forward, EMA, shuffle-BN key
forward, fused logits+CE, enqueue, full backward, gradient all-reduce, Adam.  clips/sec = 2*B*W / step time.
`value` times steps whose inputs are already resident in HBM; `e2e` times the same public-API call fed from pinned
host memory (H2D of every step's 403 MB block inside the timed region, prefetched on a copy stream, plus a D2H read
of the loss every step).  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CFG = dict(network="s3d", dim=128, K=2048, m=0.999, T=0.07, B=32, seq_len=32, img=128)
# bounded CPU sample of the workload (reference arm and cpu_baseline leg): 4 clip pairs of 16 frames = 4 of the benchmark's
# 32-frame clips per step, ~1 s per step on 16 host cores -> ~10 s for the default 8 timed steps
CPU_SAMPLE_BATCH, CPU_SAMPLE_T = 4, 16
GFLOP_PER_PAIR = {"s3d": 91.46, "s3dg": 91.46, "r50": 231.67}  # SURVEY.md 8d: q fwd+dgrad+wgrad, k fwd (conv MACs x2), one clip pair
NET_NAME = {"s3d": "S3D", "s3dg": "S3D-G", "r50": "R2D3D-50"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=8, help="timed training steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="coclr_b200", choices=["coclr_b200", "reference"])
    ap.add_argument("--precision", default="parity", choices=["parity", "mixed", "fast"])
    ap.add_argument("--net", default=CFG["network"], choices=["s3d", "s3dg", "r50"],
                    help="backbone: s3d = BASELINE.json configs 1-4 (headline), r50 = config 5 (ResNet2d3d-50), "
                         "s3dg = S3D with feature gating (select_backbone.py:8-9; same conv FLOPs)")
    ap.add_argument("--batch", type=int, default=CFG["B"])
    ap.add_argument("--seq_len", type=int, default=CFG["seq_len"])
    ap.add_argument("--moco-k", type=int, default=CFG["K"], help="queue length: 2048 = config 2 (headline), 16384 = config 3")
    ap.add_argument("--model", default="infonce", choices=["infonce", "coclr"],
                    help="infonce = configs 1-3,5; coclr = config 4 (2-stream co-training step: q fwd+bwd, k fwd, frozen "
                         "sampler fwd, top-k mined positives)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the first step")
    ap.add_argument("--no-mixed", action="store_true",
                    help="skip the extra `--precision mixed` measurement reported under config.mixed_precision")
    ap.add_argument("--no-stock-gpu", action="store_true", help="skip the stock-PyTorch-on-this-GPU baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="print the per-kernel time table of one step to stderr")
    ap.add_argument("--timeline", action="store_true",
                    help="per-phase CUDA-event timeline of one step (ms since step start, max over ranks) in the JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, logits, targets, queue, a fixed sample of the "
                         "encoder_q parameters and gradient) as DIR/<name>.npy, rank 0 only; the inputs depend only on "
                         "the arguments and the training step sums in a fixed order, so repeated runs write the same "
                         "arrays and two builds can be compared output for output")
    return ap.parse_args()


def _positive(v):
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError("must be >= 1")
    return n


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.15)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm restated in oracle/ (the Python reference itself cannot travel to the GPU box)
# ------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may really use: the cgroup CPU quota when there is one (oversubscribing it makes
    the CPU arm several times slower), else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    env = int(os.environ.get("COCLR_CPU_THREADS", "0"))
    return env if env > 0 else n


def cpu_oracle_clips_per_s(batch, seq_len, img, K, steps, warmup, net="s3d"):
    from oracle import coclr_oracle as O
    torch.set_num_threads(usable_cores())
    torch.manual_seed(0)
    sd = O.synth_state(O.infonce_shapes(128, K, network=net), seed=0)
    for k in O.param_keys(sd, "encoder_q."):
        sd[k].requires_grad_(True)
    state = {}
    g = torch.Generator().manual_seed(1)
    times = []
    for it in range(warmup + steps):
        block = torch.randn(batch, 2, 3, seq_len, img, img, generator=g)
        t0 = time.perf_counter()
        idx = torch.randperm(batch)
        logits, labels = O.infonce_forward(sd, [block], idx)
        loss = O.infonce_loss(logits[0], labels)
        qkeys = O.param_keys(sd, "encoder_q.")
        grads = torch.autograd.grad(loss, [sd[k] for k in qkeys])
        O.adam_step({k: sd[k] for k in qkeys}, dict(zip(qkeys, grads)), state)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    # clips are counted in units of the benchmark's 32-frame clip: a pair of `seq_len`-frame clips is
    # 2 * seq_len / 32 of them (conv work is linear in the number of frames)
    return 2.0 * batch * (seq_len / float(CFG["seq_len"])) / med, med


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch, sample_T = CPU_SAMPLE_BATCH, CPU_SAMPLE_T
    steps = args.steps
    val, med = cpu_oracle_clips_per_s(batch, sample_T, CFG["img"], args.moco_k, steps, 1, args.net)
    line = {"impl": "reference", "metric": "clips/sec %s InfoNCE (32x128^2, K=%d)" % (NET_NAME[args.net], args.moco_k), "value": val, "unit": "clips/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "InfoNCE %s moco-k=%d 128^2 full train step (fwd+bwd+Adam), bounded sample: "
                                   "%d clip pair(s) of %d frames per step, scaled to 32-frame clips" % (NET_NAME[args.net], args.moco_k, batch, sample_T),
                       "batch_per_step": batch, "sample_seq_len": sample_T},
            "cpu_baseline": {"value": val, "unit": "clips/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "oracle port of the reference (torch CPU fp32), %d timed steps of %d pair(s) of "
                                       "%d-frame 128^2 clips after 1 warm-up, counted as %d/32 clips each; the reference "
                                       "is pure Python and cannot travel to the GPU box" % (steps, batch, sample_T, sample_T)},
            "e2e": {"value": val, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


DUMP_MAX_ELEMS = 1 << 21     # per array: the six arrays of a dump stay under 64 MB whatever the shapes


def dump_outputs(path, outputs):
    """np.save every tensor of `outputs` (name -> tensor) as `path`/<name>.npy, float64 kept, everything else as float32.
    A tensor of more than DUMP_MAX_ELEMS elements is flattened and sampled at sorted positions drawn from a fixed seed:
    the same positions in every run with the same shapes."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t.to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32)
        np.save(os.path.join(path, name + ".npy"), t.numpy())


# ------------------------------------------------------------------------------------------------
# parity of the benched configuration: the FIRST training step of the run against the oracle (checker only; nothing
# of oracle/ is on the timed path).  Works for any world size: rank 0 simulates the W-rank world (shuffle-BN
# permutation, per-rank BatchNorm, global enqueue) in float64 from the gathered inputs and the pre-step state.
# ------------------------------------------------------------------------------------------------
def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def parity_first_step(model, run_step, block, world, rank, dev):
    import torch.distributed as dist
    from oracle import coclr_oracle as O
    sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    seed = 4242
    torch.manual_seed(seed)              # rank 0 draws the shuffle-BN permutation from the CPU RNG (pretrain.py:112)
    logits, loss = run_step(block)
    torch.cuda.synchronize()
    if world > 1:
        blocks_all = torch.empty((world,) + tuple(block.shape), dtype=block.dtype, device=dev)
        dist.all_gather_into_tensor(blocks_all, block.contiguous())
        logits_all = torch.empty((world,) + tuple(logits.shape), dtype=logits.dtype, device=dev)
        dist.all_gather_into_tensor(logits_all, logits.detach().contiguous())
    else:
        blocks_all, logits_all = block[None], logits.detach()[None]
    out = None
    store = dist.distributed_c10d._get_default_store() if world > 1 else None
    if rank != 0 and store is not None:
        store.wait(["coclr_parity_done"])     # sleep in the store client instead of spinning next to rank 0's oracle run
    if rank == 0:
        t0 = time.perf_counter()
        prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            sdd = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in sd0.items()}
            for k in O.param_keys(sdd, "encoder_q."):
                sdd[k].requires_grad_(True)
            torch.manual_seed(seed)
            idx = torch.randperm(block.shape[0] * world).to(dev)
            ref_logits, labels = O.infonce_forward(sdd, [blocks_all[r].double() for r in range(world)], idx,
                                                   keep_graph=False)
            e_logits = max(_rel(logits_all[r], ref_logits[r]) for r in range(world))
            ref_loss = float(O.infonce_loss(ref_logits[0], labels.to(dev)))
            e_queue = _rel(model.queue, sdd["queue"])
            out = {"oracle": "oracle/coclr_oracle.py in float64 on the same GPU, simulated %d-rank world" % world,
                   "step": "first training step of this run (B=%d per rank)" % block.shape[0],
                   "logits_rel_err": e_logits, "loss": float(loss), "loss_oracle": ref_loss,
                   "loss_rel_err": abs(float(loss) - ref_loss) / max(1.0, abs(ref_loss)),
                   "queue_rel_err": e_queue, "queue_ptr": [int(model.queue_ptr), int(sdd["queue_ptr"])],
                   "tolerance": 1e-3, "seconds": None}
            out["ok"] = bool(e_logits < 1e-3 and out["loss_rel_err"] < 1e-3 and e_queue < 1e-3 and
                             out["queue_ptr"][0] == out["queue_ptr"][1])
            del sdd, ref_logits
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
        torch.cuda.synchronize()
        out["seconds"] = round(time.perf_counter() - t0, 2)
        if store is not None:
            store.set("coclr_parity_done", "1")
    del blocks_all, logits_all, sd0
    torch.cuda.empty_cache()
    return out


def replicas_identical(model, world, dev):
    """Bit-exact comparison of every rank's parameters and queue (an order-independent 64-bit checksum of the raw bits)."""
    import torch.distributed as dist
    cs = torch.stack([model.encoder_q.store.flat.view(torch.int32).to(torch.int64).sum(),
                      model.encoder_k.store.flat.view(torch.int32).to(torch.int64).sum(),
                      model.queue.contiguous().view(torch.int32).to(torch.int64).sum()])
    if world == 1:
        return True
    allc = torch.empty(world, 3, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allc, cs)
    return bool((allc == allc[0:1]).all())


# ------------------------------------------------------------------------------------------------
# the same training step in stock PyTorch ops (the oracle's restatement of the reference, cuDNN / cuBLAS) on THIS GPU:
# what the unmodified reference would reach on a B200 -- "the Blackwell kernels to beat" (SURVEY.md 2a / 8d).
# fp32-strict is the arithmetic the 1e-3 parity bar needs; TF32 is PyTorch's default (misses the bar by ~40x).
# ------------------------------------------------------------------------------------------------
def stock_gpu_baseline(batch, seq_len, img, K, net, dev, steps=3):
    from oracle import coclr_oracle as O
    out = {"impl": "oracle ops in stock PyTorch %s / cuDNN %s on the same GPU" % (torch.__version__, torch.backends.cudnn.version()),
           "batch": batch, "steps": steps, "unit": "clips/s"}
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        for mode in ("fp32", "tf32"):
            torch.backends.cudnn.allow_tf32 = mode == "tf32"
            torch.backends.cuda.matmul.allow_tf32 = mode == "tf32"
            torch.backends.cudnn.benchmark = True
            sd = {k: v.to(dev) for k, v in O.synth_state(O.infonce_shapes(128, K, network=net), seed=0).items()}
            qkeys = O.param_keys(sd, "encoder_q.")
            for k in qkeys:
                sd[k].requires_grad_(True)
            state = {}
            block = torch.randn(batch, 2, 3, seq_len, img, img, device=dev)

            def step():
                idx = torch.randperm(batch).to(dev)
                logits, labels = O.infonce_forward(sd, [block], idx)
                loss = O.infonce_loss(logits[0], labels.to(dev))
                grads = torch.autograd.grad(loss, [sd[k] for k in qkeys])
                O.adam_step({k: sd[k] for k in qkeys}, dict(zip(qkeys, grads)), state)
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"ms_per_step": ms, "value": 2.0 * batch / (ms * 1e-3)}
            del sd, state, block
            torch.cuda.empty_cache()
    except Exception as ex:  # pragma: no cover
        out["error"] = repr(ex)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = prev
    return out


# ------------------------------------------------------------------------------------------------
# roofline of the dominant kernel (coclr_conv_igemm) from per-launch CUDA events of one step
# ------------------------------------------------------------------------------------------------
def conv_flops(cv):
    """Algorithmic FLOPs of one coclr_conv_igemm launch (2 x MACs of the convolution it implements)."""
    if cv.g.transposed:   # dgrad: one MAC per (dy pixel, tap, cin, cout) of the forward conv
        pix = cv.B * cv.src.T * cv.src.H * cv.src.W
        return 2.0 * pix * cv.N * cv.g.kt * cv.g.kh * cv.g.kw * cv.src.C
    pix = cv.B * cv.Td * cv.Hd * cv.Wd
    if cv.src.C == 16 and cv.g.kh == 4 and cv.g.kw == 4:   # space-to-depth stem: the (kt,7,7)x3 conv it implements
        return 2.0 * pix * cv.N * cv.g.kt * 147
    cin = 3 if cv.src.C == 8 else cv.src.C   # RGB input padded to 8 channels when the s2d stem is off
    return 2.0 * pix * cv.N * cv.g.kt * cv.g.kh * cv.g.kw * cin


def wgrad_flops(wg):
    pix = wg.B * wg.Td * wg.Hd * wg.Wd
    if wg.src.C == 16 and wg.g.kh == 4 and wg.g.kw == 4:   # space-to-depth stem: count the (kt,7,7)x3 conv it implements
        return 2.0 * pix * wg.Cout * wg.g.kt * 147
    return 2.0 * pix * wg.Cout * wg.g.kt * wg.g.kh * wg.g.kw * wg.Cin_real


def kernel_breakdown(run_step):
    from coclr_b200.engine import EncoderEngine
    from model.pretrain import InfoNCE
    EncoderEngine.profile = []
    InfoNCE.overlap_key_branch = False      # per-kernel durations are only meaningful without stream overlap
    try:
        run_step()
        torch.cuda.synchronize()
        prof = EncoderEngine.profile
    finally:
        EncoderEngine.profile = None
        InfoNCE.overlap_key_branch = True
    table = {}
    for name, a, e0, e1 in prof:
        ms = e0.elapsed_time(e1)
        t = table.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0.0})
        t["launches"] += 1
        t["ms"] += ms
        if name == "coclr_conv_igemm":
            t["flops"] += conv_flops(a[0]._obj)
        elif name == "coclr_conv_wgrad":
            t["flops"] += wgrad_flops(a[0]._obj)
    return table, prof


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, ...) write to fd 1; the contract is ONE JSON line on stdout. Point fd 1 at
    stderr for the run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from model.pretrain import InfoNCE, CoCLR
    from coclr_b200 import moco, lib as L

    B, T, HW, K = args.batch, args.seq_len, CFG["img"], args.moco_k
    coclr = args.model == "coclr"
    torch.manual_seed(0)                                   # main_nce.py:97-99
    if coclr:
        model = CoCLR(args.net, CFG["dim"], K, CFG["m"], CFG["T"], topk=5, precision=args.precision).to(dev).train()
        model.sampler.eval()                               # main_coclr.py:363
        model.queue_label.fill_(1)                         # a full queue: the top-k mining and the optimizer step run (:400-406)
        model.queue_vname.copy_(torch.arange(K, device=dev) % 997)
    else:
        model = InfoNCE(args.net, CFG["dim"], K, CFG["m"], CFG["T"], precision=args.precision).to(dev).train()
    opt = moco.FlatAdam(model.encoder_q, lr=1e-3, weight_decay=1e-5)
    gen = torch.Generator().manual_seed(1000 + rank)
    nblk = 2 if coclr else 1                               # CoCLR reads two blocks per sample (clip 1 and clip 2, RGB + flow)
    host_blocks = [torch.randn(nblk * B, 2, 3, T, HW, HW, generator=gen).pin_memory() for _ in range(2)]
    dev_blocks = [hb.to(dev) for hb in host_blocks]       # 2 x 403 MB > 126 MB L2: inputs never L2-resident
    vname = torch.randint(0, 997, (B,), device=dev)
    loss_keep = [None, None, None]                         # loss, logits, labels (InfoNCE) / positive mask (CoCLR)

    def train_step(block):
        if coclr:
            import main_coclr
            logits, target = model(block[:B], block[B:], vname)
            loss = main_coclr.multi_nce_loss(logits, target)
        else:
            logits, target = model(block)
            loss = moco.nce_cross_entropy(logits, target)
        opt.zero_grad()
        loss.backward()
        opt.step()
        loss_keep[0], loss_keep[1], loss_keep[2] = loss, logits, target
        return loss

    # ---- parity of this configuration, before anything is timed (all ranks take part; rank 0 runs the oracle) ----
    parity = None
    if not args.no_parity and not coclr:
        parity = parity_first_step(model, lambda blk: (train_step(blk), loss_keep[1], loss_keep[0])[1:], dev_blocks[0],
                                   world, rank, dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident inputs ----
    for i in range(args.warmup):
        train_step(dev_blocks[i % 2])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = L.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host = time.perf_counter()
    for i in range(args.steps):
        train_step(dev_blocks[i % 2])
    host_ms = (time.perf_counter() - t_host) * 1e3 / args.steps   # host time to ENQUEUE one step (no sync inside)
    e1.record()
    barrier()
    launches = (L.LAUNCHES - l0) // max(1, args.steps)
    same_replicas = replicas_identical(model, world, dev)
    ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    final_loss = float(loss_keep[0].detach())
    value = 2.0 * B * world / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss_keep[0].reshape(1), "logits": loss_keep[1],
                                         ("mask" if coclr else "labels"): loss_keep[2], "queue": model.queue,
                                         "encoder_q_params": model.encoder_q.store.flat,
                                         "encoder_q_grad": model.encoder_q.store.grad})

    # ---- end to end: pinned host inputs, H2D inside the timed region (prefetched), loss read back every step ----
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream()
        stage = [torch.empty_like(dev_blocks[0]) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[i % 2])          # the step that last used this buffer has finished
                stage[i % 2].copy_(host_blocks[i % 2], non_blocking=True)
                ready[i % 2].record(copy_stream)

        # the loss of every step is read back inside the timed region through pinned memory; the read of step i is
        # completed after step i + 1 has been enqueued (the way a training loop logs), so that the host keeps one
        # step ahead of the device instead of draining the pipeline with a blocking .item() after every step
        loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ready = [torch.cuda.Event() for _ in range(2)]

        def e2e_loop(n):
            for d in done:
                d.record()
            prefetch(0)
            seen = []
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[i % 2])
                loss = train_step(stage[i % 2])
                done[i % 2].record()
                loss_host[i % 2].copy_(loss.detach().reshape(1), non_blocking=True)    # D2H read of the step's result
                loss_ready[i % 2].record()
                if i >= 1:
                    loss_ready[(i - 1) % 2].synchronize()
                    seen.append(float(loss_host[(i - 1) % 2]))
            loss_ready[(n - 1) % 2].synchronize()
            seen.append(float(loss_host[(n - 1) % 2]))
            return seen
        e2e_loop(max(1, args.warmup // 2))
        barrier()
        t0 = time.perf_counter()
        e2e_loop(args.steps)
        barrier()
        dt = (time.perf_counter() - t0) / args.steps
        tt = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": 2.0 * B * world / float(tt), "unit": "clips/s",
               "h2d_bytes_per_step": host_blocks[0].numel() * 4, "d2h_bytes_per_step": 4}
        del stage
        torch.cuda.empty_cache()
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- per-phase timeline of one step (events on the streams the phases run on) ----
    timeline = None
    if args.timeline:
        moco.TIMELINE = []
        t_start = torch.cuda.Event(enable_timing=True)
        barrier()
        t_start.record()
        train_step(dev_blocks[0])
        moco.mark("step:end")
        torch.cuda.synchronize()
        tl = [(name, t_start.elapsed_time(ev)) for name, ev in moco.TIMELINE]
        moco.TIMELINE = None
        vals = torch.tensor([v for _, v in tl], device=dev)
        if world > 1:
            dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        timeline = {name: round(float(v), 3) for (name, _), v in zip(tl, vals)}

    # ---- roofline of the dominant kernel, measured live with CUDA events around every launch of one step ----
    table, prof = kernel_breakdown(lambda: train_step(dev_blocks[0]))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    cv = table.get("coclr_conv_igemm", {"ms": 0.0, "flops": 0.0, "launches": 0})
    wg = table.get("coclr_conv_wgrad", {"ms": 0.0, "flops": 0.0, "launches": 0})
    passes = 3 if args.precision == "parity" else None
    # DRAM traffic of the heaviest coclr_conv_igemm launch of the step (Conv_2c.conv1 forward) from the committed
    # `ncu --set full` capture; its algorithmic bytes are one read of the fp16 hi/lo input planes + one fp32 write
    traffic, traffic_note = None, None
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_full_summary.json")))["ncu_r02_tma_conv2c1_fwd.ncu-rep"]
        traffic = (cap["dram__bytes_read.sum"]["value"] + cap["dram__bytes_write.sum"]["value"]) * 1e6
        traffic_note = ("bytes of ONE launch of the kernel as benched (TMA-staged): Conv_2c.conv1 forward, M=524288 N=192 "
                        "K=576, from the committed `ncu --set full` capture (profiles/r02_ncu_full_summary.json); "
                        "algorithmic = 134.2e6 (input planes, read once) + 402.7e6 (fp32 output) bytes")
    except Exception:
        pass
    achieved = cv["flops"] / (cv["ms"] * 1e-3) / 1e12 if cv["ms"] > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "coclr_conv_igemm (forward + dgrad implicit GEMM)",
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": traffic if args.net == "s3d" else None, "traffic_note": traffic_note, "peak_source": peak_src,
                "launches_per_step": cv["launches"], "ms_per_step_in_kernel": cv["ms"],
                "mode": "%s (forward %s, backward %s)" % (args.precision,
                                                        "3 MMA passes fp16 hi/lo" if args.precision != "fast" else "1 pass bf16",
                                                        "3 MMA passes fp16 hi/lo, gradient planes scaled by a per-tensor power of two"
                                                        if args.precision == "parity" else
                                                        ("1 pass fp16 on the scaled gradient planes" if args.precision == "mixed"
                                                         else "1 pass bf16")),
                "tensor_work_frac": (achieved * 3 / peak_tf) if passes else None,
                "wgrad": {"achieved": wg["flops"] / (wg["ms"] * 1e-3) / 1e12 if wg["ms"] > 0 else 0.0,
                          "ms_per_step_in_kernel": wg["ms"], "launches_per_step": wg["launches"]},
                "step_breakdown_ms": {k: round(v["ms"], 3) for k, v in sorted(table.items(), key=lambda kv: -kv[1]["ms"])}}
    if args.breakdown and rank == 0:
        for k, v in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
            print("%-24s %5d launches %9.3f ms" % (k, v["launches"], v["ms"]), file=sys.stderr)
        rows = []
        for name, a, s0, s1 in prof:
            if name in ("coclr_conv_igemm", "coclr_conv_wgrad"):
                o = a[0]._obj
                fl = conv_flops(o) if name == "coclr_conv_igemm" else wgrad_flops(o)
                msl = s0.elapsed_time(s1)
                if name == "coclr_conv_igemm":
                    desc = "M=%d N=%d K=%d tr=%d" % (o.B * o.Td * o.Hd * o.Wd, o.N, o.Kreal, o.g.transposed)
                else:
                    desc = "M=%d Cout=%d K=%d splits=%d" % (o.B * o.Td * o.Hd * o.Wd, o.Cout,
                                                           o.g.kt * o.g.kh * o.g.kw * o.src.C, o.splits)
                rows.append((msl, name, desc, fl / (msl * 1e-3) / 1e12))
            elif name in ("coclr_maxpool_fwd", "coclr_maxpool_bwd"):
                o = a[0]._obj
                rows.append((s0.elapsed_time(s1), name, "C=%d in=%dx%dx%d k=%d%d%d s=%d%d%d" % (
                    o.C, o.Ti, o.Hi, o.Wi, o.g.kt, o.g.kh, o.g.kw, o.g.st, o.g.sh, o.g.sw), 0.0))
            elif name in ("coclr_bn_bwd", "coclr_affine_split"):
                o = a[0]._obj
                rows.append((s0.elapsed_time(s1), name, "M=%d C=%d" % (o.M, o.C), 0.0))
        # conv time by pixel count of the launch (which resolution level of the network it belongs to)
        by_m = {}
        for name, a, s0, s1 in prof:
            if name == "coclr_conv_igemm":
                o = a[0]._obj
                m = o.B * o.Td * o.Hd * o.Wd
                e = by_m.setdefault(m, [0, 0.0, 0.0])
                e[0] += 1
                e[1] += s0.elapsed_time(s1)
                e[2] += conv_flops(o)
        for m in sorted(by_m, reverse=True):
            n, msl, fl = by_m[m]
            print("conv_igemm launches with M=%-9d: %3d launches %7.3f ms %7.1f TF/s" % (m, n, msl, fl / (msl * 1e-3) / 1e12),
                  file=sys.stderr)
        rows.sort(reverse=True)
        for msl, name, desc, tf in rows[:60]:
            print("%8.3f ms %-18s %-40s %7.1f TF/s" % (msl, name[6:], desc, tf), file=sys.stderr)

    # ---- the same step with the single-pass fp16 backward (`--precision mixed`): identical forward, hence identical
    #      logits / loss / queue parity; NOT the headline (see DESIGN.md section 3 "precision modes") ----
    mixed = None
    if args.precision == "parity" and not args.no_mixed and not coclr:
        del model, opt
        torch.cuda.empty_cache()
        torch.manual_seed(0)
        model = InfoNCE(args.net, CFG["dim"], K, CFG["m"], CFG["T"], precision="mixed").to(dev).train()
        opt = moco.FlatAdam(model.encoder_q, lr=1e-3, weight_decay=1e-5)
        for i in range(max(3, args.warmup)):
            train_step(dev_blocks[i % 2])
        barrier()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for i in range(args.steps):
            train_step(dev_blocks[i % 2])
        m1.record()
        barrier()
        mt = torch.tensor([m0.elapsed_time(m1) / args.steps], device=dev)
        if world > 1:
            dist.all_reduce(mt, op=dist.ReduceOp.MAX)
        mixed = {"precision": "mixed (parity forward, single-pass fp16 backward on scaled gradient planes)",
                 "ms_per_step": float(mt), "value": 2.0 * B * world / (float(mt) * 1e-3), "unit": "clips/s",
                 "note": "same logits / loss / queue as the headline; gradients within the oracle-relative budget at "
                         "random init (tests/test_infonce_gpu.py::test_other_precisions_report), a real precision cut "
                         "in well-conditioned regimes -- opt-in, not the headline"}
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            try:
                v, med = cpu_oracle_clips_per_s(CPU_SAMPLE_BATCH, CPU_SAMPLE_T, HW, K, 8, 1, args.net)
                cpu = {"value": v, "unit": "clips/s", "cores": torch.get_num_threads(), "kind": "port",
                       "sample": "oracle port (torch CPU fp32) full train step on %d pairs of %d-frame 128^2 clips "
                                 "(= %d clips of 32 frames), median of 8 timed steps after 1 warm-up, %.2f s/step"
                                 % (CPU_SAMPLE_BATCH, CPU_SAMPLE_T, 2 * CPU_SAMPLE_BATCH * CPU_SAMPLE_T // 32, med)}
            except Exception as ex:  # pragma: no cover
                cpu = {"value": None, "unit": "clips/s", "cores": torch.get_num_threads(), "kind": "port",
                       "sample": "failed: %r" % (ex,)}
        stock = None
        if not args.no_stock_gpu and world == 1 and not coclr:
            stock = stock_gpu_baseline(B, T, HW, K, args.net, dev)
        mname = "InfoNCE" if not coclr else "CoCLR 2-stream topk=5"
        line = {"metric": "clips/sec %s %s (32x128^2, K=%d)" % (NET_NAME[args.net], mname, K), "value": value, "unit": "clips/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (fp16/bf16 hi-lo split operands, fp32 accumulate)" if args.precision == "parity" else
                         ("bf16" if args.precision == "fast" else "f32 forward / bf16 backward"),
                "data": "synthetic",
                "config": {"workload": ("InfoNCE %s moco-k=%d bs=%d/GPU seq_len=%d 128^2, full train step "
                                        "(q fwd, EMA, shuffle-BN k fwd, fused logits+CE, enqueue, bwd, all-reduce, Adam)"
                                        % (NET_NAME[args.net], K, B, T)) if not coclr else
                                       ("CoCLR %s moco-k=%d topk=5 bs=%d/GPU seq_len=%d 128^2, full co-training step with a "
                                        "full queue (q fwd, EMA, shuffle-BN k fwd, frozen eval-BN sampler fwd on the second "
                                        "view, fused logits, same-source + top-k mined mask, multi-positive NCE loss, "
                                        "enqueue x2, bwd, all-reduce, Adam); 2 of the 4 clips of a sample are counted"
                                        % (NET_NAME[args.net], K, B, T)),
                           "global_batch": B * world, "parallelism": "dp%d" % world, "precision": args.precision,
                           "l2": "two alternating 403 MB input blocks per rank (> 126 MB L2)",
                           "pairs_per_s": value / 2, "final_loss": final_loss, "host_enqueue_ms_per_step": host_ms,
                           "algorithmic_tflops": value / 2 * GFLOP_PER_PAIR[args.net] * (1.25 if coclr else 1.0) * (T / 32.0) / 1e3,
                           "mixed_precision": mixed, "phase_timeline_ms": timeline},
                "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline, "parity": parity, "replicas_identical": same_replicas}
        if stock is not None:
            line["stock_gpu_baseline"] = stock
        if cpu is not None:
            line["cpu_baseline"] = cpu
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
