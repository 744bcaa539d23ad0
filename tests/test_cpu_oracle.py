"""not-gpu: the oracle restatement against the golden vectors produced by the unmodified reference, and against
stored results of the reference's own modules (tests/golden/make_reference_checks.py)."""
import json
import os

import numpy as np
import pytest
import torch

import reference_inputs as I
from oracle import fixtures
from oracle import seist_ref as R

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF = np.load(os.path.join(GOLD, "reference_checks.npz"))


@pytest.mark.parametrize("name", ["seist_s_dpk", "seist_m_dpk", "seist_m_emg", "seist_s_pmp", "seist_s_baz"])
def test_oracle_matches_golden(name):
    g = fixtures.load(GOLD, name)
    spec = R.spec_for(name)
    with torch.no_grad():
        y, _ = R.forward(g["state_dict"], g["x"], spec, training=False)
    assert (y - g["y_eval"]).abs().max().item() <= 2e-5 * g["y_eval"].abs().max().item()
    if name != "seist_s_dpk":
        return      # one full backward on CPU is enough for the time budget
    sd = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v)
          for k, v in g["state_dict"].items()}
    y, bufs = R.forward(sd, g["x"], spec, training=True)
    loss = R.bce_loss(y, g["target"])
    loss.backward()
    assert abs(loss.item() - g["loss"].item()) <= 1e-5 * abs(g["loss"].item())
    gmax = max(v.abs().max().item() for v in g["grads"].values())
    for k, ref in g["grads"].items():
        assert (sd[k].grad - ref).abs().max().item() <= 1e-4 * ref.abs().max().item() + 1e-6 * gmax, k
    for k, b in g["buffers_after"].items():
        assert (bufs[k].float() - b.float()).abs().max().item() <= 1e-5 * (b.float().abs().max().item() + 1e-3), k


def test_oracle_matches_reference_modules():
    """Train mode, drop rates zeroed: the oracle against the output of the reference's modules on the same parameters."""
    for name in I.MODULE_MODELS:
        sd, x = I.module_inputs(name)
        assert np.array_equal(I.probe(x.numpy()), REF[f"modules.{name}.x_probe"]), "seeded input changed"
        y_ref = torch.from_numpy(REF[f"modules.{name}.y"])
        y, _ = R.forward(sd, x, R.spec_for(name), training=True)
        assert torch.allclose(y, y_ref, atol=1e-6), name


def test_pad_and_sizes():
    # _auto_pad_1d semantics (SURVEY §3.5)
    assert R.auto_pad_amounts(8192, 11, 2) == (4, 5)
    assert R.auto_pad_amounts(8192, 15, 2) == (6, 7)
    assert R.auto_pad_amounts(8192, 19, 2) == (8, 9)
    assert R.auto_pad_amounts(4096, 7, 1) == (3, 3)
    for L in (1000, 1001, 6000, 8192):
        for k, s in ((11, 2), (7, 2), (5, 1), (3, 1)):
            l, r = R.auto_pad_amounts(L, k, s)
            assert (L + l + r - k) // s + 1 == -(-L // s)
    assert R.upsampling_sizes(128, 8192, 6) == [256, 512, 1024, 2048, 4096, 8192]
    assert R.upsampling_sizes(94, 6000, 6) == [187, 375, 750, 1501, 3001, 6000]
    assert R.head_layers(R.spec_for("seist_m_dpk")) == [(96, 64, 7), (64, 32, 7), (32, 24, 7), (24, 16, 7),
                                                         (16, 16, 7), (16, 6, 11)]


@pytest.mark.parametrize("name", I.DROPOUT_MODELS)
def test_dropout_sites_and_rates_match_reference_modules(name):
    """Every nn.Dropout / timm DropPath of the unmodified reference model (site = module path, rate = .p / .drop_prob,
    models/seist.py:114,228,239,360-366,446,470,484; linspace schedule :705) must appear in the compiled plan as the
    drop factor of the op that absorbs it, with the same probability — and the plan must not drop anywhere else."""
    from seist_b200 import _lib
    from seist_b200 import plan as P
    from seist_b200.models import create_model
    with open(os.path.join(GOLD, "reference_dropout_sites.json")) as f:
        ref_sites = json.load(f)[name]          # [module path, rate] of the reference model's modules
    expect = {}
    for path, p in ref_sites:
        head, leaf = path.rsplit(".", 1)
        site = {
            "droppath0": (head + ".proj", "p_path"),
            "droppath1": (head + ".mlp.lin1", "p_path"),
            "dropout": (head + ".lin1", "p_elem"),                 # MLP.dropout (head ends with .mlp)
            "k_dropout": (head + ".k_proj", "p_elem"),
            "attn_dropout": (head + ".core", "p_attn"),
            "proj_dropout": (head + ".out_proj", "p_elem"),
            "attn_droppath": (head + ".attention.out_proj", "p_path"),
            "gconv_droppath": (head + ".gconv.mlp.lin1", "p_alpha"),
            "mlp_droppath": (head + ".mlp.lin1", "p_path"),
        }[leaf]
        assert site not in expect, site
        expect[site] = p
    m = create_model(name, in_channels=3, in_samples=1024).train()
    flat = P.FlatState(m, torch.device("cpu"))
    plan = P.PlanBuilder(m, flat, 2, 1024, True).build()
    got = {}
    for op in plan.fwd_ops:
        if op.kind not in (_lib.CONV_FWD, _lib.ATT_FWD):
            continue
        for field in ("p_elem", "p_path", "p_alpha", "p_attn"):
            v = float(getattr(op, field))
            if v > 0 or (op.name, field) in expect:
                got[(op.name, field)] = v
    missing = {k: v for k, v in expect.items() if abs(got.get(k, 0.0) - v) > 1e-7}
    extra = {k: v for k, v in got.items() if v > 0 and k not in expect}
    assert not missing, list(missing.items())[:8]
    assert not extra, list(extra.items())[:8]
    assert sum(1 for v in expect.values() if v > 0) >= 20
