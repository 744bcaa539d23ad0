"""-m gpu: the public API (create_model / forward / loss / backward) against the golden vectors the
unmodified reference produced (tests/golden/make_golden.py) and against the oracle on fresh inputs.

Tolerances (BASELINE.json north_star): outputs within 1e-3 relative (max-abs normalised) of the
reference's CPU fp32 forward; P/S argmax indices bit-exact; gradients within 2e-3 of each tensor's
max-abs with an absolute floor of 1e-5 x the largest gradient (several reference gradients are
analytically zero — conv bias in front of BatchNorm, key bias under softmax — and hold only noise)."""
import os

import pytest
import torch

from oracle import fixtures
from oracle import seist_ref as R
from seist_b200.models import BCELoss, HuberLoss, create_model

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ZERO = dict(path_drop_rate=0, attn_drop_rate=0, key_drop_rate=0, mlp_drop_rate=0, other_drop_rate=0)


def _load(name):
    g = fixtures.load(GOLD, name)
    m = create_model(name, in_channels=3, in_samples=g["x"].shape[-1])
    m.load_state_dict(g["state_dict"], strict=True)
    return g, m.cuda()


def _detection_edges_match(y, ref, tol=1, amb=2e-3):
    """SURVEY §8c: the detection channel (0) has plateaus and exact ties, so it is compared through the end points
    of its > 0.5 intervals, +-`tol` samples.  Edges where the reference itself is within `amb` of the threshold in
    the neighbourhood are ambiguous under a 1e-3 output tolerance and skipped."""
    def edges(v):
        m = (v > 0.5).int()
        return (m[1:] - m[:-1]).nonzero().flatten() + 1
    for n in range(ref.shape[0]):
        ea, eb = edges(y[n, 0]), edges(ref[n, 0])
        for src, dst, base in ((eb, ea, ref[n, 0]), (ea, eb, ref[n, 0])):
            for i in src.tolist():
                lo, hi = max(i - 2, 0), min(i + 2, base.numel())
                if (base[lo:hi] - 0.5).abs().min().item() < amb:
                    continue
                if dst.numel() == 0 or (dst - i).abs().min().item() > tol:
                    return False
    return True


def _check_grads(model, ref_grads, rtol=2e-3, floor=1e-5):
    gmax = max(v.abs().max().item() for v in ref_grads.values())
    bad = []
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        ref = ref_grads[k]
        err = (p.grad.cpu() - ref).abs().max().item()
        if err > rtol * ref.abs().max().item() + floor * gmax:
            bad.append((k, err, ref.abs().max().item()))
    assert not bad, bad[:10]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["seist_s_dpk", "seist_m_dpk", "seist_m_emg", "seist_s_pmp", "seist_s_baz"])
def test_eval_matches_reference_golden(name):
    g, m = _load(name)
    m.eval()
    with torch.no_grad():
        y = m(g["x"].cuda()).cpu()
    ref = g["y_eval"]
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
    if name.endswith("dpk"):
        assert torch.equal(y[:, 1:].argmax(-1), ref[:, 1:].argmax(-1))   # P and S picks bit-exact
        assert _detection_edges_match(y, ref)                             # detection intervals, +-1 sample


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["seist_s_dpk", "seist_m_dpk", "seist_m_emg", "seist_s_pmp", "seist_s_baz"])
def test_train_step_matches_reference_golden(name):
    g, m = _load(name)
    m.set_drop_rates(**ZERO)
    m.train()
    y = m(g["x"].cuda())
    ref = g["y_train"]
    assert (y.detach().cpu() - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
    if name.endswith("dpk"):
        loss = BCELoss(weight=[[0.5], [1], [1]])(y, g["target"].cuda())
    elif name.endswith("pmp"):
        from seist_b200.models.loss import CELoss
        loss = CELoss(weight=[1, 1])(y, g["target"].cuda())          # fused CUDA CE (config.py:147-155)
    else:
        loss = HuberLoss()(y, g["target"].cuda())
    assert abs(loss.item() - g["loss"].item()) <= 1e-4 * abs(g["loss"].item())
    loss.backward()
    _check_grads(m, g["grads"])
    sd = m.state_dict()
    for k, b in g["buffers_after"].items():
        if k.endswith("num_batches_tracked"):
            assert int(sd[k]) == int(b), k
        else:
            assert (sd[k].cpu() - b).abs().max().item() <= 1e-3 * (b.abs().max().item() + 1e-3), k


@pytest.mark.gpu
def test_l_model_and_batch_against_oracle():
    """seist_l_dpk (no fixture): random non-degenerate parameters, train mode, oracle on the same inputs."""
    from harness import randomize
    torch.manual_seed(0)
    m = randomize(create_model("seist_l_dpk", in_channels=3, in_samples=4096), seed=3)
    m.set_drop_rates(**ZERO)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    x, tgt = R.synth_waveforms(3, 4096, seed=11)
    sd_g = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v)
            for k, v in sd.items()}
    y_ref, _ = R.forward(sd_g, x, R.spec_for("seist_l_dpk"), training=True)
    loss_ref = R.bce_loss(y_ref, tgt)
    loss_ref.backward()
    m = m.cuda().train()
    y = m(x.cuda())
    assert (y.detach().cpu() - y_ref.detach()).abs().max().item() <= 1e-3 * y_ref.abs().max().item()
    loss = BCELoss(weight=[[0.5], [1], [1]])(y, tgt.cuda())
    loss.backward()
    assert abs(loss.item() - loss_ref.item()) <= 1e-4 * abs(loss_ref.item())
    _check_grads(m, {k: sd_g[k].grad for k, _ in m.named_parameters()})


@pytest.mark.gpu
def test_dropout_is_active_and_reproducible_for_a_fixed_counter():
    """Dropout/DropPath are not bit-matched to torch's Philox stream (SURVEY §4.4): they are active, draw new masks
    every training forward and are exactly reproducible when the engine's step counter is restored.  The mask
    semantics (rates, 1/keep scaling, per-sample DropPath) are pinned in test_gpu_parity2.py."""
    g, m = _load("seist_s_dpk")
    m.train()
    x = g["x"].cuda()
    eng = m.engine()
    with torch.no_grad():
        y0 = m(x)
        seed = eng.dropout_seed()
        y1 = m(x)
        assert not torch.equal(y0, y1)        # a new step -> new masks
        eng.set_dropout_seed(seed - 1)
        y2 = m(x)
        assert torch.equal(y0, y2)            # same counter value -> same masks
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(x), m(x))        # eval: identity
    assert torch.isfinite(y1).all()


@pytest.mark.gpu
def test_cpu_input_fails_loudly():
    m = create_model("seist_s_dpk", in_channels=3, in_samples=1024)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 1024))


@pytest.mark.gpu
def test_full_size_batch_properties():
    """BASELINE.json's full configuration — seist_m_dpk on (512, 3, 8192) — through size-independent properties
    (the oracle needs minutes at this size): eval mode is per-waveform independent, so rows of the full batch
    must equal the same rows run as a small batch (catches 32-bit index / byte-offset overflow: the arena is
    ~11 GB here); a training step is reproducible for a fixed dropout seed and yields finite, non-trivial
    gradients for every parameter; the BatchNorm batch statistics of the full batch equal the count-weighted
    combination of two half batches (linearity of the fused statistic sums)."""
    from seist_b200.train import Trainer
    g, m = _load("seist_m_dpk")
    L, N = 8192, 512
    x, tgt = R.synth_waveforms(N, L, seed=5)
    x, tgt = x.cuda(), tgt.cuda()
    m.eval()
    with torch.no_grad():
        y_full = m(x)
        idx = torch.tensor([0, 1, 255, 256, 510, 511], device="cuda")
        y_rows = m(x[idx].contiguous())
    assert y_full.shape == (N, 3, L) and torch.isfinite(y_full).all()
    assert float(y_full.min()) >= 0.0 and float(y_full.max()) <= 1.0
    assert (y_full[idx] - y_rows).abs().max().item() <= 2e-6
    assert torch.equal(y_full[idx][:, 1:].argmax(-1), y_rows[:, 1:].argmax(-1))
    # eval of a small batch at this length against the reference golden restatement (CPU oracle, seconds)
    y_ref, _ = R.forward(g["state_dict"], x[idx[:2]].cpu(), R.spec_for("seist_m_dpk"), training=False)
    assert (y_rows[:2].cpu() - y_ref).abs().max().item() <= 1e-3 * y_ref.abs().max().item()

    # training step: reproducible under a fixed seed, finite gradients everywhere
    m.train()
    eng = m.engine()
    loss_fn = BCELoss(weight=[[0.5], [1], [1]])

    def step():
        for p in m.parameters():
            p.grad = None
        y = m(x)
        loss = loss_fn(y, tgt)
        loss.backward()
        return loss.detach().clone(), torch.cat([p.grad.flatten() for p in m.parameters()]).clone()

    m(x[:2].contiguous())                 # creates the engine's dropout counter
    seed = eng.dropout_seed()
    l0, g0 = step()
    eng.set_dropout_seed(seed)            # the forward advances the counter: rewind to replay the same masks
    l1, g1 = step()
    assert torch.isfinite(l0) and torch.isfinite(g0).all()
    assert abs(l0.item() - l1.item()) <= 1e-6 * abs(l0.item())
    # atomically accumulated sums are order-dependent in the last bits: compare to float tolerance
    assert (g0 - g1).abs().max().item() <= 1e-4 * g0.abs().max().item()
    assert float((g0 != 0).float().mean()) > 0.9

    # BN statistic sums are linear in the batch: mean over the full batch == average of the half-batch means
    m.set_drop_rates(**ZERO)
    sd0 = {k: v.clone() for k, v in g["state_dict"].items()}

    key = "stem.0.convs.0.norm.running_mean"

    def stem_mean(xb):
        m.load_state_dict(sd0, strict=True)
        with torch.no_grad():
            m(xb)
        after = m.state_dict()[key].clone()
        return (after - 0.9 * sd0[key].cuda()) / 0.1      # momentum 0.1 (reference default): recover the batch mean

    mu_full, mu_a, mu_b = stem_mean(x), stem_mean(x[:N // 2].contiguous()), stem_mean(x[N // 2:].contiguous())
    # recovering the batch mean from the momentum update amplifies the fp32 rounding of running_mean 10x
    tol = 1e-5 * (mu_full.abs().max().item() + 1e-3) + 2e-6 * (sd0[key].abs().max().item() + 1e-3)
    assert (mu_full - 0.5 * (mu_a + mu_b)).abs().max().item() <= tol


@pytest.mark.gpu
def test_trainer_prefetch_equals_direct_step():
    """Trainer.prefetch() + step() (copy stream, one batch ahead) must train exactly like step(x, target)."""
    import copy
    from seist_b200.train import Trainer
    g, m = _load("seist_s_dpk")
    m2 = copy.deepcopy(m)
    x, tgt = g["x"], g["target"]
    xp, tp = x.pin_memory(), tgt.pin_memory()
    ta, tb = Trainer(m, lr=1e-3), Trainer(m2, lr=1e-3)
    la = [float(ta.step(x.cuda(), tgt.cuda())) for _ in range(3)]
    lb = [float(tb.step(xp, tp))]
    for _ in range(2):
        tb.prefetch(xp, tp)
        lb.append(float(tb.step()))
    # float atomics make the weight gradients order-dependent in the last bits and Adam amplifies that: 2e-4
    assert all(abs(a - b) <= 2e-4 * abs(a) for a, b in zip(la, lb)), (la, lb)
    assert la[2] != la[0]                                  # the parameters really moved
    with pytest.raises(RuntimeError):
        tb.step()                                          # nothing staged


@pytest.mark.gpu
def test_inference_graph_equals_eval_forward():
    """§8f-4: the captured forward-only plan reproduces model.eval()(x) bit for bit, batch after batch, and equals the golden."""
    from seist_b200.infer import InferenceGraph
    g, m = _load("seist_s_dpk")
    m.eval()
    x = g["x"].cuda()
    with torch.no_grad():
        want = m(x).clone()
    ig = InferenceGraph(m, x.shape[0], x.shape[2])
    assert torch.equal(ig(x), want)
    x2 = torch.roll(x, 1, 0)
    assert (ig(x2) - torch.roll(want, 1, 0)).abs().max().item() <= 2e-6    # per-waveform independent in eval mode
    assert torch.equal(ig(x.cpu().pin_memory()).clone(), want)   # pinned host input
    ref = g["y_eval"]
    assert (ig(x).cpu() - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
    with pytest.raises(ValueError):
        ig(x[:1])
