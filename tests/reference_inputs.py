"""Seeded inputs of the comparisons against the reference's own code whose results are stored in
tests/golden/reference_checks.npz (written by tests/golden/make_reference_checks.py).  The tests and the generator
build the inputs here, so both see the same values."""
import numpy as np
import torch

MODULE_MODELS = ("seist_s_dpk", "seist_l_emg", "seist_s_pmp")
MODULE_L = 2048
DROPOUT_MODELS = ("seist_s_dpk", "seist_m_dpk", "seist_l_dpk", "seist_m_emg")
PICK_CASES = ((1, 50), (3, 50), (5, 8), (2, 200))
PICK_THRESHOLDS = (0.3, 0.05)
LABEL_L = 2048
CODA_RATIO = 1.4
LABEL_CASES = (([300], [700]), ([5], [60]), ([1900], [2040]), ([], []), ([100, 900], [400, 1300]), ([800], []), ([], [500]),
               ([2047], [2047 + 30]), ([0], [3]))


def probe(a):
    """A strided sample of an input array, stored beside the results to pin the random stream that made it."""
    a = np.asarray(a).reshape(-1)
    return a[::max(1, a.size // 512)].copy()


def module_inputs(name):
    """Non-degenerate parameters (random-init train output is nearly flat) and a batch of two waveforms."""
    from harness import randomize
    from seist_b200.models import create_model
    seed = MODULE_MODELS.index(name)
    m = randomize(create_model(name, in_channels=3, in_samples=MODULE_L), seed=100 + seed)
    x = torch.randn(2, 3, MODULE_L, generator=torch.Generator().manual_seed(200 + seed))
    return m.state_dict(), x


def pick_traces(topk, mpd, n=48, L=2048):
    """Random Gaussian bumps plus noise, scaled into [0, 1), and four crafted rows."""
    rng = np.random.default_rng(topk * 100 + mpd)
    t = np.arange(L, dtype=np.float32)
    x = np.zeros((n, L), dtype=np.float32)
    for i in range(n):
        for _ in range(rng.integers(0, 6)):
            c, w, a = rng.integers(0, L), rng.uniform(3, 40), rng.uniform(0.1, 1.0)
            x[i] += a * np.exp(-((t - c) ** 2) / (2 * w * w)).astype(np.float32)
        x[i] = x[i] + 0.02 * rng.standard_normal(L).astype(np.float32)
        # no clipping: equal peak heights have no defined order in the reference (np.argsort's default sort is unstable)
        x[i] = (x[i] - x[i].min()) / max(1.0, float(x[i].max() - x[i].min()) * 1.01)
    x[0] = 0.0                          # no peak at all
    x[1, :] = 0.5                       # flat above the threshold: no rising edge
    x[2] = 0.0
    x[2, 100:110] = 0.8                 # flat-topped peak: rising edge only
    x[3] = 0.0
    x[3, 0], x[3, -1] = 0.9, 0.9        # first / last samples cannot be peaks
    return x


def normalize_inputs():
    """(mode, x) per normalisation mode; x has a constant channel (scale 0 -> 1)."""
    rng = np.random.default_rng(0)
    out = []
    for mode in ("std", "max", ""):
        x = rng.standard_normal((3, 4096)).astype(np.float32) * 3 + 1
        x[1] = 2.5
        out.append((mode, x))
    return out


def label_cases():
    """(shape, width, case index, P picks, S picks) of the dpk soft-label comparison."""
    return [(shape, width, ci, ppks, spks) for shape in ("gaussian", "triangle", "box") for width in (25, 50, 11)
            for ci, (ppks, spks) in enumerate(LABEL_CASES)]
