"""not-gpu: host logic — registry/checkpoint surface, parameter tree, plan compiler (through the CPU
interpreter, end to end against the reference's golden vectors), C-ABI library symbols."""
import ctypes
import os

import pytest
import torch

from oracle import fixtures
from oracle import seist_ref as R
from oracle.plan_interp import Interp, keep_mask, rng_u16
from seist_b200 import _lib
from seist_b200 import plan as P
from seist_b200 import models
from seist_b200.models import create_model, get_model_list, register_model
from seist_b200.models.seist import dpk_up_sizes, same_pad, split_mptl, split_msmc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ZERO = dict(path_drop_rate=0, attn_drop_rate=0, key_drop_rate=0, mlp_drop_rate=0, other_drop_rate=0)


def test_registry_surface():
    names = get_model_list()
    assert len(names) == 15 and "seist_m_dpk" in names
    with pytest.raises(ValueError):
        create_model("no_such_model")
    with pytest.raises(Exception):
        register_model(models.seist.seist_s_dpk)
    with pytest.raises(TypeError):          # the reference passes these explicitly -> duplicate kwarg
        create_model("seist_m_dpk", path_drop_rate=0.0)
    for n in ("BCELoss", "BinaryFocalLoss", "CELoss", "CombinationLoss", "FocalLoss", "HuberLoss", "MousaviLoss",
              "MSELoss", "save_checkpoint", "load_checkpoint"):
        assert hasattr(models, n)


@pytest.mark.parametrize("name", ["seist_s_dpk", "seist_m_dpk", "seist_m_emg"])
def test_state_dict_matches_reference_checkpoint(name):
    g = fixtures.load(GOLD, name)
    m = create_model(name, in_channels=3, in_samples=8192)
    sd = m.state_dict()
    assert list(sd.keys()) == list(g["state_dict"].keys())
    for k, v in g["state_dict"].items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, k
    m.load_state_dict(g["state_dict"], strict=True)
    assert [k for k, _ in m.named_parameters()] == list(g["grads"].keys())


def test_checkpoint_roundtrip(tmp_path):
    m = create_model("seist_s_emg", in_channels=3, in_samples=1024)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    path = str(tmp_path / "ck.pth")
    models.save_checkpoint(path, 3, m, opt, 0.5)
    ck = models.load_checkpoint(path, torch.device("cpu"))
    assert ck["epoch"] == 3 and not ck["use_ddp"] and not ck["use_compile"]
    m2 = create_model("seist_s_emg", in_channels=3, in_samples=1024)
    m2.load_state_dict(ck["model_dict"], strict=True)


def test_channel_arithmetic():
    assert split_msmc(24, 3, 2) == [16, 8] and split_msmc(64, 4, 2) == [32, 32] and split_msmc(96, 3, 2) == [64, 32]
    assert split_mptl(24, 0.6, 8) == (16, 8) and split_mptl(16, 0.6, 8) == (16, 0) and split_mptl(96, 0.6, 32) == (64, 32)
    assert same_pad(8192, 11, 2) == (4, 5) and same_pad(1001, 7, 2) == (3, 3)
    assert dpk_up_sizes(94, 6000, 6) == [187, 375, 750, 1501, 3001, 6000]
    with pytest.raises(AssertionError):
        same_pad(100, 1, 2)


def test_plan_compiler_end_to_end_vs_reference_golden():
    """Forward tape, derived backward, accumulate flags and the BN-backward algebra, executed by the CPU
    interpreter, reproduce the reference's outputs, gradients and running statistics."""
    g = fixtures.load(GOLD, "seist_s_dpk")
    m = create_model("seist_s_dpk", in_channels=3, in_samples=8192)
    m.load_state_dict(g["state_dict"], strict=True)
    m.set_drop_rates(**ZERO)
    x = g["x"][:2]
    flat = P.FlatState(m, torch.device("cpu"))
    pl = P.PlanBuilder(m, flat, 2, 8192, training=False).build()
    P.allocate(pl, False)
    y = Interp(pl).run_fwd(x)
    assert (y - g["y_eval"][:2]).abs().max().item() < 1e-4
    # train mode on the full fixture batch (statistics depend on the batch)
    x = g["x"]
    pl = P.PlanBuilder(m, flat, x.shape[0], 8192, training=True).build()
    P.allocate(pl, True)
    it = Interp(pl)
    y = it.run_fwd(x).clone()
    assert (y - g["y_train"]).abs().max().item() < 1e-4
    p = y.clone().requires_grad_(True)
    R.bce_loss(p, g["target"]).backward()
    it.run_bwd(p.grad)
    gmax = max(v.abs().max().item() for v in g["grads"].values())
    for k, ref in g["grads"].items():
        err = (flat.grad_view(k) - ref).abs().max().item()
        assert err <= 1e-3 * ref.abs().max().item() + 1e-6 * gmax, (k, err)
    sd = m.state_dict()
    for k, b in g["buffers_after"].items():
        assert (sd[k].float() - b.float()).abs().max().item() <= 1e-3 * (b.float().abs().max().item() + 1e-3), k


def test_plan_compiler_regression_head_vs_reference_golden():
    """Same as above for the regression family (seist_m_emg: HEADVEC ops, scaled sigmoid, Huber loss)."""
    g = fixtures.load(GOLD, "seist_m_emg")
    m = create_model("seist_m_emg", in_channels=3, in_samples=8192)
    m.load_state_dict(g["state_dict"], strict=True)
    m.set_drop_rates(**ZERO)
    x = g["x"]
    flat = P.FlatState(m, torch.device("cpu"))
    pl = P.PlanBuilder(m, flat, x.shape[0], 8192, training=False).build()
    P.allocate(pl, False)
    y = Interp(pl).run_fwd(x)
    y = y if y.dim() == 2 else y[:, :, 0]
    assert (y - g["y_eval"]).abs().max().item() < 1e-4 * max(1.0, g["y_eval"].abs().max().item())
    pl = P.PlanBuilder(m, flat, x.shape[0], 8192, training=True).build()
    P.allocate(pl, True)
    it = Interp(pl)
    y = it.run_fwd(x).clone()
    y2 = y if y.dim() == 2 else y[:, :, 0]
    assert (y2 - g["y_train"]).abs().max().item() < 1e-4 * max(1.0, g["y_train"].abs().max().item())
    p = y2.clone().requires_grad_(True)
    R.huber_loss(p, g["target"]).backward()
    it.run_bwd(p.grad.reshape(y.shape))
    gmax = max(v.abs().max().item() for v in g["grads"].values())
    for k, ref in g["grads"].items():
        err = (flat.grad_view(k) - ref).abs().max().item()
        assert err <= 1e-3 * ref.abs().max().item() + 1e-6 * gmax, (k, err)


ALL_VARIANTS = [f"seist_{size}_{task}" for size in "sml" for task in ("dpk", "pmp", "emg", "baz", "dis")]


@pytest.mark.parametrize("name,L", [(n, 2048 if n == "seist_s_pmp" else 1024) for n in ALL_VARIANTS])
def test_plan_compiler_vs_oracle_random_cotangent(name, L):
    """All 15 registered variants (detection/picking, classification with softmax, the three regression heads; S, M
    and the L preset with 4-branch MSMC and two MPTL blocks): random non-degenerate parameters, train mode,
    arbitrary output cotangent - the interpreter must reproduce the pinned oracle's outputs and parameter gradients."""
    from harness import randomize
    torch.manual_seed(0)
    m = randomize(create_model(name, in_channels=3, in_samples=L), seed=7)
    m.set_drop_rates(**ZERO)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    x, _ = R.synth_waveforms(3, L, seed=2)
    sd_g = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone())
            for k, v in sd.items()}
    y_ref, _ = R.forward(sd_g, x, R.spec_for(name), training=True)
    dy = torch.randn(y_ref.shape, generator=torch.Generator().manual_seed(5)) / y_ref.numel()
    y_ref.backward(dy)
    flat = P.FlatState(m, torch.device("cpu"))
    pl = P.PlanBuilder(m, flat, 3, L, training=True).build()
    P.allocate(pl, True)
    it = Interp(pl)
    y = it.run_fwd(x).clone()
    y2 = y.reshape(y_ref.shape)
    assert (y2 - y_ref.detach()).abs().max().item() <= 1e-4 * max(1e-3, y_ref.abs().max().item())
    it.run_bwd(dy.reshape(y.shape))
    grads = {k: sd_g[k].grad for k, _ in m.named_parameters()}
    gmax = max(v.abs().max().item() for v in grads.values())
    for k, ref in grads.items():
        err = (flat.grad_view(k) - ref).abs().max().item()
        assert err <= 1e-3 * ref.abs().max().item() + 1e-5 * gmax, (k, err)


def test_grad_combine_plan_equals_default_plan(monkeypatch):
    """GRAD_COMBINE (opt-in, SEIST_COMBINE_CIN): the compiler marks the wide 1x1 convs, emits the in-place BN
    backward before their three backward ops and re-points those ops at the combined gradient; executed by the
    interpreter the parameter gradients must equal the default plan's (reference golden batch, train mode)."""
    g = fixtures.load(GOLD, "seist_s_dpk")
    x = g["x"][:2, :, :2048].contiguous()
    tgt = g["target"][:2, :, :2048].contiguous()

    def grads(thr):
        monkeypatch.setenv("SEIST_COMBINE_CIN", thr)
        m = create_model("seist_s_dpk", in_channels=3, in_samples=2048)
        m.load_state_dict(g["state_dict"], strict=True)
        m.set_drop_rates(**ZERO)
        flat = P.FlatState(m, torch.device("cpu"))
        pl = P.PlanBuilder(m, flat, 2, 2048, training=True).build()
        P.allocate(pl, True)
        it = Interp(pl)
        y = it.run_fwd(x).clone()
        p = y.clone().requires_grad_(True)
        R.bce_loss(p, tgt).backward()
        it.run_bwd(p.grad)
        return pl, flat.G.clone()

    p0, g0 = grads("0")
    p1, g1 = grads("8")
    n_comb = sum(op.kind == _lib.GRAD_COMBINE for op in p1.bwd_ops)
    assert not any(op.kind == _lib.GRAD_COMBINE for op in p0.bwd_ops) and n_comb > 20
    assert len(p1.bwd_ops) == len(p0.bwd_ops) + n_comb
    assert (g1 - g0).abs().max().item() <= 1e-5 * g0.abs().max().item()


def test_plan_structure_and_sync_points():
    m = create_model("seist_m_dpk", in_channels=3, in_samples=8192)
    flat = P.FlatState(m, torch.device("cpu"))
    pl = P.PlanBuilder(m, flat, 2, 8192, training=True, world=2).build()
    assert len(pl.bns) == 115          # SURVEY §0.2: 115 BatchNorm layers in seist_m_dpk
    fwd_sync = sorted(b for op in pl.fwd_ops for b in op.sync_bn)
    chained = {e.idx for e in pl.bns if e.is_chained}
    assert fwd_sync == sorted(set(range(115)) - chained)   # every BN's statistics reduced exactly once
    bwd_sync = sorted(b for op in pl.bwd_ops for b in op.sync_bn)
    assert bwd_sync == fwd_sync
    # BN-input elements per waveform match the survey's byte model (E_BN = 1 869 824)
    e_bn = folded = 0
    for op in pl.fwd_ops:
        if op.kind == _lib.CONV_FWD and op.out.bn >= 0:
            e_bn += op.out.C * op.out.L
            if pl.bns[op.out.bn].chain >= 0:      # attention.norm on top of aggr.norm: folded, never materialised
                folded += op.out.C * op.out.L
    assert e_bn + folded == 1869824 and folded == 11264


def test_rng_reference_values():
    import numpy as np
    v = rng_u16(7, 3, np.arange(8, dtype=np.uint64))
    assert v.dtype == np.uint32 and int(v.max()) < 65536 and len(set(v.tolist())) >= 7
    # drop rate of the 16-bit lanes: p = 0.2 over 2^20 draws, scaled survivors keep the mean at ~1
    m = keep_mask(0.2, 11, 5, np.arange(1 << 20, dtype=np.uint64))
    assert abs(float((m == 0).float().mean()) - 0.2) < 2e-3 and abs(float(m.mean()) - 1.0) < 3e-3


def test_library_exports_every_declared_symbol():
    assert os.path.isfile(_lib.LIB_PATH), "build first: python __graft_entry__.py"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in _lib.EXPORTS:
        assert hasattr(lib, sym), sym
    hdr = open(os.path.join(os.path.dirname(_lib.LIB_PATH), "..", "..", "include", "seist_b200.h")).read()
    import re
    declared = set(re.findall(r"\b(seist_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    L = _lib.lib()      # ABI version + struct layout checks (no GPU needed)
    assert L.seist_abi_version() == _lib.ABI_VERSION


def test_cyclic_lr_matches_torch_scheduler():
    """Trainer's host-side schedule must equal torch.optim.lr_scheduler.CyclicLR as the reference configures it
    (training/train.py:343-354: exp_range, cycle_momentum=False, gamma = base_lr ** (1 / (2 * steps)))."""
    from seist_b200.train import cyclic_lr
    base, mx, up, down, steps = 8e-5, 1e-3, 20, 30, 120
    gamma = base ** ((steps * 2) ** -1)
    for mode, g in (("triangular", None), ("exp_range", gamma)):
        p = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.Adam([p], lr=base)
        sch = torch.optim.lr_scheduler.CyclicLR(opt, base_lr=base, max_lr=mx, step_size_up=up, step_size_down=down,
                                                mode=mode, gamma=gamma if g else 1.0, cycle_momentum=False)
        for it in range(steps):
            ref = opt.param_groups[0]["lr"]
            assert abs(cyclic_lr(it, base, mx, up, down, g) - ref) <= 1e-9 + 1e-7 * ref, (mode, it)
            opt.step()
            sch.step()
