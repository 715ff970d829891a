"""CPU-side checks: C-ABI library builds/loads/exports every declared symbol, the nn.Module surface has
the reference's state_dict keys, the engine graph covers exactly the reference's parameters, and the product
refuses to run without CUDA (no CPU fallback)."""
import ctypes
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_all_header_symbols():
    from coclr_b200 import build, lib, _signatures
    path = build.build()
    assert os.path.exists(path)
    cdll = lib.load()
    header = open(os.path.join(ROOT, "include", "coclr_b200.h")).read()
    declared = set(re.findall(r"\b(coclr_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(cdll, name), "library does not export %s" % name
    assert declared == set(_signatures.EXPORTS), declared ^ set(_signatures.EXPORTS)


def test_library_is_sm100a_tcgen05():
    import subprocess
    from coclr_b200 import build
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    assert "UTCHMMA" in sass and "LDTM" in sass and "UBLKCP" in sass


def test_state_dict_keys_match_reference_surface():
    from model.pretrain import InfoNCE, UberNCE, CoCLR
    from oracle import coclr_oracle as O
    m = InfoNCE("s3d", 128, 128)
    want = set(O.with_aliases(O.synth_state(O.infonce_shapes(128, 128))).keys())
    have = set(m.state_dict().keys())
    assert want == have, (sorted(want - have)[:5], sorted(have - want)[:5])
    assert len(list(m.encoder_q.parameters())) == 235
    assert not any(p.requires_grad for p in m.encoder_k.parameters())
    u = UberNCE("s3d", 128, 128)
    assert "queue_label" in u.state_dict()
    c = CoCLR("s3d", 128, 128, topk=5)
    for k in ("queue_second", "queue_vname", "queue_label", "sampler.0.Conv_1a.conv1.weight", "sampler.4.bias"):
        assert k in c.state_dict(), k
    assert c.queue_is_full is False
    # call sites written against the DDP-wrapped reference model keep working (main_coclr.py:363,403)
    assert c.module is c and c.module.queue_is_full is False and c.module.sampler is c.sampler
    assert not any(k.startswith("module.") for k in c.state_dict())
    # a checkpoint saved from the reference's DDP-wrapped model ('module.' prefix, main_nce.py:271-279) loads as is
    ddp_style = {"module." + k: v.clone() for k, v in m.state_dict().items()}
    ddp_style["module.queue_ptr"] = torch.tensor([24])
    m2 = InfoNCE("s3d", 128, 128)
    m2.load_state_dict(ddp_style, strict=True)
    assert int(m2.queue_ptr) == 24 and m2._ptr() == 24
    assert torch.equal(m2.encoder_q[0].Conv_2c.conv1.weight, m.encoder_q[0].Conv_2c.conv1.weight)


def test_select_backbone_contract():
    from backbone.select_backbone import select_backbone
    m, p = select_backbone("s3d")
    assert p == {"feature_size": 1024}
    with pytest.raises(NotImplementedError):
        select_backbone("nope")
    mg, pg = select_backbone("s3dg")      # S3D with feature gating (reference select_backbone.py:8-9)
    assert pg == {"feature_size": 1024} and mg.gating
    extra = set(dict(mg.named_parameters())) - set(dict(m.named_parameters()))
    assert len(extra) == 2 * 4 * 9 and all(".gating_b" in k for k in extra)   # (weight, bias) x 4 branches x 9 blocks
    assert tuple(mg.Mixed_4b.gating_b1.fc.weight.shape) == (208, 208)


def test_s3dg_graph_and_plan_dry_run():
    """S3D-G: parameter layout equals the reference's (through the oracle's shape table, itself checked against the
    reference's state_dict in tests/test_oracle.py), and the launch plan gates every SepInception output: forward
    mean -> 4 fc -> apply after the block's BatchNorm, backward reduce -> 4 fc_bwd -> apply before its BatchNorm backward."""
    from coclr_b200 import lib as L
    from coclr_b200.engine import Graph, ParamStore, EncoderEngine
    from coclr_b200.s3d_spec import s3d_stages
    from oracle import coclr_oracle as O
    g = Graph(s3d_stages(3, gating=True), 3, head_dim=128, bb_prefix="0.")
    lay = dict(g.param_layout())
    shapes = {k[len("encoder_q."):]: tuple(v) for k, v in O.infonce_shapes(128, 128, network="s3dg").items()
              if k.startswith("encoder_q.") and (k.endswith(".weight") or k.endswith(".bias"))}
    assert set(lay) == set(shapes) and all(tuple(lay[k]) == s for k, s in shapes.items())
    L.DRY_RUN = True
    try:
        st = ParamStore(g, torch.device("cpu"))
        eng = EncoderEngine(st, g, "parity")
        p = eng.plan(2, 8, 64, 64, True, True)
        fw = [fn.__name__ for fn, _ in p.fwd]
        assert fw.count("coclr_gate_mean") == 9 and fw.count("coclr_gate_fc") == 36 and fw.count("coclr_gate_apply") == 9
        for i, n in enumerate(fw):
            if n == "coclr_gate_mean":
                assert fw[i - 1] == "coclr_affine_split" and fw[i + 1:i + 6] == ["coclr_gate_fc"] * 4 + ["coclr_gate_apply"]
        bw = [fn.__name__ for fn, _ in p.bwd]
        assert bw.count("coclr_gate_bwd_reduce") == 9 and bw.count("coclr_gate_fc_bwd") == 36
        for i, n in enumerate(bw):
            if n == "coclr_gate_bwd_reduce":
                assert bw[i + 1:i + 7] == ["coclr_gate_fc_bwd"] * 4 + ["coclr_gate_bwd_apply", "coclr_bn_bwd"]
        assert p.bwd_split is None       # the gating parameters are reduced with everything else at the end
        # every gating parameter's gradient is written by exactly one launch
        base = st.grad.data_ptr()
        offs = sorted((a[4].value - base) // 4 for fn, a in p.bwd if fn.__name__ == "coclr_gate_fc_bwd")
        want = sorted(st.offsets[k][0] for k in st.offsets if k.endswith(".fc.weight"))
        assert offs == want and len(set(offs)) == 36
        # the forward-only plan (key encoder) gates too
        pk = eng.plan(2, 8, 64, 64, True, False)
        assert [fn.__name__ for fn, _ in pk.fwd].count("coclr_gate_apply") == 9
    finally:
        L.DRY_RUN = False


def test_graph_covers_reference_parameters():
    from coclr_b200.engine import Graph
    from coclr_b200.s3d_spec import s3d_stages
    from oracle import coclr_oracle as O
    g = Graph(s3d_stages(3), 3, head_dim=128, bb_prefix="0.")
    lay = dict(g.param_layout())
    shapes = {k[len("encoder_q."):]: tuple(v) for k, v in O.infonce_shapes(128, 128).items()
              if k.startswith("encoder_q.") and (k.endswith(".weight") or k.endswith(".bias"))}
    assert set(lay) == set(shapes)
    for k, s in shapes.items():
        assert tuple(lay[k]) == s, k
    bufs = dict(g.buffer_layout())
    rm = {k[len("encoder_q."):-len(".running_mean")]: v[0] for k, v in O.infonce_shapes(128, 128).items()
          if k.startswith("encoder_q.") and k.endswith(".running_mean")}
    assert bufs == rm
    # 77 backbone convs (the 9 pairs of branch-opening 1x1 convs may run as one launch each), 13 pools (SURVEY.md appendix A)
    assert sum(len(it.weight_names) for k, it in g.items if k == "conv") == 77
    assert sum(1 for k, _ in g.items if k == "pool") == 13
    # shapes at 32 x 128^2
    dims = g.backbone_out.dims_fn((32, 128, 128))
    assert dims == (4, 4, 4) and g.backbone_out.C == 1024


def test_no_cpu_fallback():
    from model.pretrain import InfoNCE
    m = InfoNCE("s3d", 128, 128)
    with pytest.raises(Exception) as ei:
        m(torch.zeros(2, 2, 3, 8, 64, 64))
    assert "CUDA" in str(ei.value)


def test_oracle_not_imported_by_product():
    import subprocess
    out = subprocess.run(["grep", "-rIl", "-E", r"^\s*(from|import) +oracle", os.path.join(ROOT, "coclr_b200"),
                          os.path.join(ROOT, "model"), os.path.join(ROOT, "backbone")], capture_output=True, text=True)
    assert out.stdout.strip() == ""


def test_launch_plans_build_on_cpu_dry_run():
    """Structure of the forward/backward launch lists (built over CPU tensors, never run): every tensor gets
    a gradient, op counts match the architecture, first-writer/accumulate flags are consistent."""
    from coclr_b200 import lib as L
    from coclr_b200.engine import Graph, ParamStore, EncoderEngine
    from coclr_b200.s3d_spec import s3d_stages
    L.DRY_RUN = True
    try:
        g = Graph(s3d_stages(3), 3, head_dim=128, bb_prefix="0.")
        st = ParamStore(g, torch.device("cpu"))
        eng = EncoderEngine(st, g, "parity")
        p = eng.plan(2, 8, 64, 64, True, True)
        names = [fn.__name__ for fn, _ in p.fwd]
        fused = 9 if g.fuse_b12 else 0    # per SepInception: branch1.0 + branch2.0 1x1 convs run as one conv, one BN pass
        assert names.count("coclr_conv_igemm") == 77 - fused + 2
        assert names.count("coclr_maxpool_fwd") == 13
        assert names.count("coclr_affine_split") == (77 - 9 * 3) - fused + 2   # one fused BN-finalize+apply+split per tensor (concat tensors hold 4 BNs) + 2 head splits
        bn = [fn.__name__ for fn, _ in p.bwd]
        assert bn.count("coclr_conv_wgrad") + bn.count("coclr_conv_wgrad_s2d") == 77 - fused + 2   # the stem's runs in space-to-depth form
        assert bn.count("coclr_conv_igemm") == 76 - fused + 2   # no dgrad for the RGB stem conv
        assert bn.count("coclr_maxpool_bwd") == 13
        assert bn.count("coclr_bn_bwd") == 77 - 9 * 3 - fused
        # fused 1x1 convs: member weights / BN parameters adjacent in the flat buffer, consumers read channel slices
        for kind, it in g.items:
            if kind == "conv" and len(it.weight_names) == 2:
                w = st.view_span([n + ".weight" for n in it.weight_names])
                assert w.shape[0] == sum(it.couts) and w.data_ptr() == st.view(it.weight_names[0] + ".weight").data_ptr()
        for t in g.tensors:     # per-tensor BatchNorm: members tile the channels in order, parameters follow that order
            if t.bn_members:
                assert [m[1] for m in t.bn_members] == sorted(m[1] for m in t.bn_members), t.name
                assert sum(m[2] for m in t.bn_members) == t.C and t.bn_members[0][1] == 0
                offs = [st.offsets[m[0] + ".weight"][0] for m in t.bn_members]
                assert offs == sorted(offs) and offs[-1] - offs[0] == sum(m[2] for m in t.bn_members[:-1]), t.name
        sliced = [it for kind, it in g.items if kind == "conv" and it.src_C != it.src.C and it.src is not g.input]
        assert len(sliced) == 2 * fused and all(it.src_coff % 8 == 0 and it.src_C % 8 == 0 for it in sliced)
        g0 = Graph(s3d_stages(3), 3, head_dim=128, bb_prefix="0.", fuse_b12=False)
        assert [n for n, _ in g0.param_layout()] != [] and sorted(n for n, _ in g0.param_layout()) == sorted(n for n, _ in g.param_layout())
        # inference plan has no gradient buffers
        p2 = eng.plan(2, 8, 64, 64, True, False)
        assert not p2.bwd and all(a.grad is None for a in p2.acts.values())
        # flat layout: every BN group contiguous, every offset 16-byte aligned
        assert all(off % 4 == 0 for off, _, _ in st.offsets.values())
    finally:
        L.DRY_RUN = False


def test_r50_plan_structure_dry_run():
    """ResNet2d3d-50 launch lists (SURVEY.md row a14): 53 backbone convs, residual wiring, gradient coverage."""
    from coclr_b200 import lib as L
    from coclr_b200.engine import Graph, ParamStore, EncoderEngine
    from coclr_b200.r50_spec import r50_stages
    from oracle import coclr_oracle as O
    L.DRY_RUN = True
    try:
        g = Graph(r50_stages(3), 3, head_dim=128, feature_size=2048, bb_prefix="0.")
        assert g.stem_s2d
        st = ParamStore(g, torch.device("cpu"))
        want = {k[len("encoder_q."):]: tuple(v) for k, v in O.infonce_shapes(128, 128, network="r50").items()
                if k.startswith("encoder_q.") and (k.endswith(".weight") or k.endswith(".bias"))}
        assert {k: tuple(v[2]) for k, v in st.offsets.items()} == want
        eng = EncoderEngine(st, g, "parity")
        p = eng.plan(2, 8, 64, 64, True, True)
        assert p.backbone_out.dims == (4, 2, 2) and p.backbone_out.spec.C == 2048
        names = [fn.__name__ for fn, _ in p.fwd]
        assert names.count("coclr_conv_igemm") == 53 + 2
        assert names.count("coclr_maxpool_fwd") == 1
        assert names.count("coclr_affine_split") == 53 + 2
        bn = [fn.__name__ for fn, _ in p.bwd]
        assert bn.count("coclr_conv_wgrad") + bn.count("coclr_conv_wgrad_s2d") == 53 + 2
        assert bn.count("coclr_conv_igemm") == 52 + 2
        assert bn.count("coclr_bn_bwd") == 53
        res = [t for t in g.tensors if t.residual is not None]
        assert len(res) == 16 and sum(1 for t in res if t.residual.name.endswith(".ds")) == 4
    finally:
        L.DRY_RUN = False


@pytest.mark.parametrize("stem", ["s3d", "r50"])
def test_space_to_depth_stem_is_the_same_convolution(stem):
    """Host logic of the space-to-depth stem (EncoderEngine._make_s2d + the layout coclr_pack_input_s2d writes): the
    stride-1 (kt,4,4) conv over 2x2-blocked pixels with the gathered weight equals the reference's stride-2 (kt,7,7)
    conv (backbone/s3dg.py:145 Conv_1a.conv1; backbone/resnet_2d3d.py:138 conv1), and the scatter-back of its weight
    gradient equals the original conv's weight gradient.  Pure torch on the CPU."""
    import torch.nn.functional as F
    from coclr_b200 import lib as L
    from coclr_b200.engine import Graph, ParamStore, EncoderEngine
    from coclr_b200.s3d_spec import s3d_stages
    from coclr_b200.r50_spec import r50_stages
    L.DRY_RUN = True
    try:
        if stem == "s3d":
            g = Graph(s3d_stages(3), 3, head_dim=None)
            name, k, s, p = "Conv_1a.conv1", (1, 7, 7), (1, 2, 2), (0, 3, 3)
        else:
            g = Graph(r50_stages(3), 3, head_dim=None, feature_size=2048)
            name, k, s, p = "conv1", (5, 7, 7), (2, 2, 2), (2, 3, 3)
        st = ParamStore(g, torch.device("cpu"))
        eng = EncoderEngine(st, g, "parity")
    finally:
        L.DRY_RUN = False
    gen = torch.Generator().manual_seed(3)
    w = st.view(name + ".weight")
    w.copy_(torch.randn(w.shape, generator=gen) * 0.1)
    eng._refresh_s2d()
    d = eng.s2d[name]
    w_eff = d["w_eff"].clone().requires_grad_(True)                 # [64, 12, kt, 4, 4]
    B, T, H, W = 2, 6, 16, 12
    x = torch.randn(B, 3, T, H, W, generator=gen)
    # what coclr_pack_input_s2d writes: out[b, t, Y, X, (dy*2+dx)*Cin + c] = x[b, c, t, 2Y+dy, 2X+dx]
    xs = x.view(B, 3, T, H // 2, 2, W // 2, 2).permute(0, 4, 6, 1, 2, 3, 5).reshape(B, 12, T, H // 2, W // 2)
    wr = w.detach().clone().requires_grad_(True)
    y_ref = F.conv3d(x, wr, stride=s, padding=p)
    y_s2d = F.conv3d(xs, w_eff, stride=(s[0], 1, 1), padding=(p[0], 2, 2))[:, :, :, :H // 2, :W // 2]
    assert y_ref.shape == y_s2d.shape
    assert float((y_ref - y_s2d).abs().max()) < 1e-4 * float(y_ref.abs().max())
    # backward: gradient w.r.t. the gathered weight, scattered back the way _s2d_wgrad_op does
    dy = torch.randn(y_ref.shape, generator=gen)
    y_ref.backward(dy)
    y_s2d.backward(dy)
    dw = torch.zeros(wr.numel()).index_add_(0, d["idx"], w_eff.grad.reshape(-1) * d["mask"]).view_as(wr)
    assert float((dw - wr.grad).abs().max()) < 1e-4 * float(wr.grad.abs().max())
    # the map is one-to-one on the 7x7 taps: every original weight is used exactly once
    used = torch.zeros(wr.numel()).index_add_(0, d["idx"], d["mask"])
    assert torch.equal(used, torch.ones_like(used))


GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_cli_accepts_every_reference_flag():
    """Drop-in command line: every option of the reference's main_nce.py / main_coclr.py (tests/golden/reference_cli.json,
    made by tests/golden/make_golden_cli.py) parses here, with the same default for the options that shape the hot path."""
    import json
    import importlib.util

    def load(name):     # this repository's script by path (the reference has files of the same name)
        spec = importlib.util.spec_from_file_location("coclr_b200_cli_" + name, os.path.join(ROOT, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    main_nce, main_coclr = load("main_nce"), load("main_coclr")
    ref = json.load(open(os.path.join(GOLDEN, "reference_cli.json")))
    assert len(ref["main_nce"]) > 30 and len(ref["main_coclr"]) > 30

    for mod, name in ((main_nce, "main_nce"), (main_coclr, "main_coclr")):
        for flag, (takes_value, nargs2) in ref[name].items():
            argv = [flag] + ((["a", "b"] if nargs2 else ["1"]) if takes_value else [])
            try:
                mod.parse_args(argv)
            except SystemExit:
                pytest.fail("%s does not accept %s" % (mod.__name__, flag))
    a = main_nce.parse_args([])
    assert (a.net, a.model, a.batch_size, a.seq_len, a.num_seq, a.img_dim, a.lr, a.wd) == ("s3d", "infonce", 32, 32, 2, 128, 1e-3, 1e-5)
    assert (a.moco_dim, a.moco_k, a.moco_m, a.moco_t, a.schedule) == (128, 2048, 0.999, 0.07, [120, 160])
    c = main_coclr.parse_args([])
    assert (c.topk, c.reverse, c.model, c.dataset) == (5, False, "coclr", "ucf101-2stream-2clip")


def test_training_losses_are_the_reference_formulas():
    """The two mask losses of the training loops as the reference computes them (tests/golden/reference_losses.npz,
    executed from the reference's own source text by tests/golden/make_golden_cli.py): multi_nce_loss
    (main_coclr.py:343-346) and the UberNCE loss lines (main_nce.py:321-322) against main_coclr.multi_nce_loss /
    main_nce.multi_label_nce_loss, bit-for-bit."""
    import importlib.util
    import numpy as np

    def load(name):
        spec = importlib.util.spec_from_file_location("coclr_b200_cli2_" + name, os.path.join(ROOT, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    main_nce, main_coclr = load("main_nce"), load("main_coclr")
    ref = np.load(os.path.join(GOLDEN, "reference_losses.npz"))
    assert len(ref["logits"]) == 3
    for logits, mask, multi, uber in zip(ref["logits"], ref["mask"], ref["multi_nce_loss"], ref["ubernce_loss"]):
        logits, mask = torch.from_numpy(logits), torch.from_numpy(mask)
        assert torch.equal(main_coclr.multi_nce_loss(logits, mask), torch.tensor(multi))
        assert torch.equal(main_nce.multi_label_nce_loss(logits, mask), torch.tensor(uber))


def _load_cli(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("coclr_b200_cli_" + name, os.path.join(ROOT, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_two_checkpoint_init_follows_reference(tmp_path):
    """main_coclr.py --pretrain A B (reference main_coclr.py:250-302): ONLY encoder_q.* of A goes into encoder_q AND
    encoder_k (A's own EMA weights, A's sampler.* -- present when A is itself a CoCLR checkpoint, i.e. from co-training
    cycle 2 on -- and all queues are dropped); ONLY encoder_q.* of B becomes the sampler."""
    main_coclr = _load_cli("main_coclr")
    from model.pretrain import CoCLR, InfoNCE
    torch.manual_seed(0)
    a = CoCLR("s3d", 128, 128, topk=5)       # first checkpoint: a CoCLR-shaped state (has sampler.* and queue_second)
    b = InfoNCE("s3d", 128, 128)             # second checkpoint: the oracle
    with torch.no_grad():
        for i, m in enumerate((a.encoder_q, a.encoder_k, a.sampler, b.encoder_q, b.encoder_k)):
            m[4].bias.fill_(float(i + 1))    # q_A=1, k_A=2, sampler_A=3 (stale), q_B=4, k_B=5
    pa, pb = str(tmp_path / "a.pth.tar"), str(tmp_path / "b.pth.tar")
    torch.save({"epoch": 7, "state_dict": {"module." + k: v for k, v in a.state_dict().items()}}, pa)   # DDP-style keys
    torch.save({"epoch": 9, "state_dict": b.state_dict()}, pb)
    state = main_coclr.two_checkpoint_state([pa, pb])
    assert not any("queue" in k for k in state)
    assert float(state["encoder_q.4.bias"][0]) == 1.0 and float(state["encoder_k.4.bias"][0]) == 1.0
    assert float(state["sampler.4.bias"][0]) == 4.0          # the oracle's encoder_q, NOT A's stale sampler (3)
    model = CoCLR("s3d", 128, 128, topk=5)
    q0 = model.queue.clone()
    res = main_coclr.load_two_checkpoints(model, [pa, pb])
    assert not res.unexpected_keys
    assert all("queue" in k for k in res.missing_keys)
    assert float(model.encoder_q[4].bias[0]) == 1.0 and float(model.encoder_k[4].bias[0]) == 1.0
    assert float(model.sampler[4].bias[0]) == 4.0
    assert torch.equal(model.encoder_k[0].Conv_2c.conv1.weight, a.encoder_q[0].Conv_2c.conv1.weight)
    assert torch.equal(model.queue, q0)                      # queues are always re-filled
    # the reference's own merge gives the same key -> source mapping: tests/golden/reference_two_checkpoint.npz holds
    # what it made of two checkpoints whose values name their own keys (tests/golden/make_golden_cli.py)
    import numpy as np
    ref = np.load(os.path.join(GOLDEN, "reference_two_checkpoint.npz"))
    pa, pb = str(tmp_path / "a_names.pth.tar"), str(tmp_path / "b_names.pth.tar")
    torch.save({"epoch": 7, "state_dict": {str(k): "first:" + str(k) for k in ref["first_keys"]}}, pa)
    torch.save({"epoch": 9, "state_dict": {str(k): "second:" + str(k) for k in ref["second_keys"]}}, pb)
    want = dict(zip(ref["merged_keys"].tolist(), ref["merged_values"].tolist()))
    assert len(want) > 2000 and main_coclr.two_checkpoint_state([pa, pb]) == want


def test_reference_adam_state_converts_to_flat(tmp_path):
    """A checkpoint written by the reference carries a torch.optim.Adam state_dict with one param group per
    named_parameter of the whole model (main_nce.py:190-200,276); resuming from it must restore the moments and the step
    count of encoder_q instead of silently restarting them.  Uses the dry-run store (no CUDA)."""
    main_nce = _load_cli("main_nce")
    from coclr_b200 import lib as L, moco
    from model.pretrain import InfoNCE
    torch.manual_seed(0)
    model = InfoNCE("s3d", 128, 128)
    params = [{"params": p} for _, p in model.named_parameters()]       # reference main_nce.py:190-198
    ref_opt = torch.optim.Adam(params, lr=1e-3, weight_decay=1e-5)
    for p in model.encoder_q.parameters():
        p.grad = torch.randn_like(p) * 1e-3
    ref_opt.step()
    ref_opt.step()
    sd = ref_opt.state_dict()
    L.DRY_RUN = True
    try:
        from coclr_b200.engine import Graph, ParamStore

        class _Enc:      # the two things load_optimizer_state needs from an encoder: named_parameters() and .store
            def __init__(self, enc):
                bb = enc[0]
                g = Graph(bb._stages, bb.input_channel, head_dim=enc.dim, feature_size=enc.feature_size, bb_prefix="0.")
                self.store, self._enc = ParamStore(g, "cpu"), enc

            def named_parameters(self):
                return self._enc.named_parameters()
        enc = _Enc(model.encoder_q)
        opt = moco.FlatAdam(enc, lr=1e-3, weight_decay=1e-5)
        assert main_nce.load_optimizer_state(opt, sd, enc, "cpu")
        assert opt.step_count == 2
        names = [n for n, _ in model.encoder_q.named_parameters()]
        for i in (0, 17, len(names) - 1):
            off, n, _ = enc.store.offsets[names[i]]
            assert torch.equal(opt.exp_avg[off:off + n], sd["state"][i]["exp_avg"].reshape(-1))
            assert torch.equal(opt.exp_avg_sq[off:off + n], sd["state"][i]["exp_avg_sq"].reshape(-1))
        assert not main_nce.load_optimizer_state(opt, None, enc, "cpu")
        assert not main_nce.load_optimizer_state(opt, {"state": {}, "param_groups": []}, enc, "cpu")
    finally:
        L.DRY_RUN = False


def test_weight_gradient_plans_cover_the_benchmark_shapes():
    """Host-side planner of the TMA-staged weight-gradient kernel (no launch, no GPU): at B=32, T=32, 128^2 every
    weight gradient of S3D -- the space-to-depth stem and the temporally strided stem conv included -- is covered,
    except the (1,3,3) convs on 4x4 frames (tiles would be more than half padding)."""
    import ctypes as C
    from coclr_b200 import lib as L, engine as E
    from coclr_b200.s3d_spec import s3d_stages
    lib = L.load()
    L.DRY_RUN = True
    try:
        g = E.Graph(s3d_stages(3), 3, head_dim=128, bb_prefix="0.")
        st = E.ParamStore(g, "cpu")
        eng = E.EncoderEngine(st, g, "parity")
        p = eng.plan(2, 32, 128, 128, True, True)     # the planner only looks at T, H, W and the channel counts
        info = (C.c_int * 8)()
        missed, kinds = [], {}
        for w in p.wgrads + p.s2d_wgrads:
            gm = w.g
            key = (gm.kt, gm.kh, gm.kw, gm.st)
            if lib.coclr_wgrad_tma_plan(C.byref(w), info) == 1:
                kinds[key] = kinds.get(key, 0) + 1
                assert info[3] in (64, 128, 192, 256) and 1 <= info[4] <= 4 and info[5] >= 2
            else:
                missed.append((key, w.Hd, w.Wd))
        assert all(k == (1, 3, 3, 1) and h == 4 for k, h, _ in missed) and len(missed) == 4, missed
        assert kinds[(1, 4, 4, 1)] == 1 and kinds[(7, 1, 1, 2)] == 1        # both stem layers
        assert kinds[(1, 3, 3, 1)] == 15 and kinds[(3, 1, 1, 1)] == 19 and kinds[(1, 1, 1, 1)] == 1 + 3 * 9 + 2
    finally:
        L.DRY_RUN = False


def test_weight_gradient_workspaces_dry_run():
    """Workspace wiring of the weight-gradient launches (host logic on the dry-run plan): the launches that go to the
    side stream share ONE workspace big enough for each of them; the space-to-depth stem's launch, which runs on the main
    stream while the side stream may still be busy, has its own; nothing overlaps."""
    import ctypes as C
    from coclr_b200 import lib as L, engine as E
    from coclr_b200.s3d_spec import s3d_stages
    lib = L.load()
    L.DRY_RUN = True
    try:
        g = E.Graph(s3d_stages(3), 3, head_dim=128, bb_prefix="0.")
        st = E.ParamStore(g, "cpu")
        eng = E.EncoderEngine(st, g, "parity")
        p = eng.plan(2, 8, 64, 64, True, True)
        assert len(p.wgrads) + len(p.s2d_wgrads) == 77 - (9 if g.fuse_b12 else 0) + 2 and len(p.s2d_wgrads) == 1
        shared = {w.ws for w in p.wgrads}
        assert len(shared) == 1 and p.wg_ws is not None and shared == {p.wg_ws.data_ptr()}
        need = [int(lib.coclr_wgrad_ws_floats(C.byref(w))) for w in p.wgrads]
        assert max(need) == p.wg_ws.numel() and all(w.ws_floats == p.wg_ws.numel() for w in p.wgrads)
        assert sum(1 for n in need if n > 0) >= 45           # all but the (1,3,3) convs on 4x4 / 2x2 frames at this shape
        own = p.s2d_wgrads[0]
        lo, hi = p.wg_ws.data_ptr(), p.wg_ws.data_ptr() + 4 * p.wg_ws.numel()
        assert own.ws and not (lo <= own.ws < hi) and own.ws_floats == int(lib.coclr_wgrad_ws_floats(C.byref(own))) > 0
        # launch accounting: a weight gradient with a workspace is two kernels
        wl = [(fn, a) for fn, a in p.bwd if fn.__name__ == "coclr_conv_wgrad"]
        assert sum(L.kernels_of(fn, a) for fn, a in wl) == len(wl) + sum(1 for n in need if n > 0)
    finally:
        L.DRY_RUN = False


def test_overlapped_allreduce_ranges_are_final_when_reduced():
    """The flat gradient is all-reduced in two parts (moco._EncodeFn.backward): the first part while the second segment
    of the backward launch list still runs.  Host logic, checked on the dry-run plan: the two range sets partition the
    buffer, and no launch of the second segment writes a gradient that the first all-reduce has already taken."""
    import ctypes as C
    from coclr_b200 import lib as L, engine as E
    from coclr_b200.s3d_spec import s3d_stages
    from coclr_b200.r50_spec import r50_stages
    L.DRY_RUN = True
    try:
        for stages, fs in ((s3d_stages(3), 1024), (r50_stages(3), 2048)):
            g = E.Graph(stages, 3, head_dim=128, feature_size=fs, bb_prefix="0.")
            st = E.ParamStore(g, "cpu")
            eng = E.EncoderEngine(st, g, "parity")
            p = eng.plan(2, 8, 64, 64, True, True)
            assert p.bwd_split is not None and 0 < p.bwd_split < len(p.bwd)
            first, rest = eng.grad_ranges(p)
            cover = sorted(first + rest)
            assert cover[0][0] == 0 and cover[-1][1] == st.numel
            assert all(a[1] == b[0] for a, b in zip(cover, cover[1:])), cover
            assert sum(hi - lo for lo, hi in first) >= 0.7 * st.numel
            base = st.grad.data_ptr()

            def written(fn, args):
                """element offsets of the flat gradient this launch writes"""
                o = args[0]._obj if (args and hasattr(args[0], "_obj")) else None
                name = fn.__name__
                out = []
                if name == "coclr_conv_wgrad":
                    out.append(o.dw)
                elif name == "coclr_conv_wgrad_s2d":
                    out.append(eng.s2d[[k for k in eng.s2d][0]]["dw"].data_ptr())
                elif name == "coclr_bn_bwd":
                    out += [o.dgamma, o.dbeta]
                elif name == "coclr_l2norm_bwd":
                    out.append(args[4].value)
                elif name == "coclr_bias_relu_bwd":
                    out.append(args[3].value)
                return [(ptr - base) // 4 for ptr in out if ptr]
            late = [off for fn, args in p.bwd[p.bwd_split:] for off in written(fn, args)]
            early = [off for fn, args in p.bwd[:p.bwd_split] for off in written(fn, args)]
            assert late and early
            assert all(any(lo <= off < hi for lo, hi in rest) for off in late), "a late launch writes an early range"
            assert all(any(lo <= off < hi for lo, hi in first) for off in early), "an early launch writes a late range"
    finally:
        L.DRY_RUN = False
