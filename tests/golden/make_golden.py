"""Generate the tests/golden/<model>.<i>.pt fixtures (oracle/fixtures.py) by executing the UNMODIFIED reference.

Run in the build container only:  python tests/golden/make_golden.py
Each fixture holds: the reference's pretrained state_dict (weights are the only pinned artefacts the
reference ships, SURVEY §0.4), seeded synthetic inputs/targets, and what the reference computes from
them: eval output, train-mode (all drop rates zeroed) output, loss, every parameter gradient, and
the post-step BN running buffers.  The oracle (oracle/seist_ref.py) and the CUDA path are both
checked against these on machines where /root/reference does not exist.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import fixtures  # noqa: E402
from oracle import reference_import as ri  # noqa: E402
from oracle import seist_ref as R  # noqa: E402

FIXTURES = [  # (model, checkpoint, batch, length)
    ("seist_s_dpk", "seist_s_dpk_diting.pth", 4, 8192),   # BASELINE.json configs[0]
    ("seist_m_dpk", "seist_m_dpk_diting.pth", 2, 8192),
    ("seist_m_emg", "seist_m_emg_diting.pth", 2, 8192),
    ("seist_s_pmp", "seist_s_pmp_diting.pth", 4, 8192),    # HeadClassification + CELoss(weight=[1, 1]) (config.py:147-155)
    ("seist_s_baz", "seist_s_baz_diting.pth", 4, 8192),    # HeadRegression x 360 + HuberLoss (config.py:167-175)
]
ONLY = set(sys.argv[1:])      # python make_golden.py seist_s_pmp seist_s_baz  -> only these (the others stay byte-identical)


def main():
    M = ri.import_reference_models()
    torch.manual_seed(0)
    torch.set_num_threads(8)
    for name, ck, n, length in FIXTURES:
        if ONLY and name not in ONLY:
            continue
        blob = torch.load(os.path.join(ri.REF_ROOT, "pretrained", ck), map_location="cpu")
        sd = blob["model_dict"] if "model_dict" in blob else blob
        model = M.create_model(name, in_channels=3, in_samples=length)
        model.load_state_dict(sd, strict=True)
        ri.zero_drop_rates(model)
        x, tgt = R.synth_waveforms(n, length, seed=20240921)
        if name.endswith("pmp"):
            cls = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(5))
            tgt = torch.nn.functional.one_hot(cls, 2).float()
        elif name.endswith("baz"):
            tgt = torch.rand(n, 1, generator=torch.Generator().manual_seed(5)) * 360.0
        elif not name.endswith("dpk"):
            tgt = torch.rand(n, 1, generator=torch.Generator().manual_seed(5)) * 8.0
        model.eval()
        with torch.no_grad():
            y_eval = model(x)
        model.train()
        y_train = model(x)
        if name.endswith("dpk"):
            loss = M.BCELoss(weight=[[0.5], [1], [1]])(y_train, tgt)
        elif name.endswith("pmp"):
            loss = M.CELoss(weight=[1, 1])(y_train, tgt)
        else:
            loss = M.HuberLoss()(y_train, tgt)
        loss.backward()
        out = {
            "model": name, "state_dict": {k: v.clone() for k, v in sd.items()},
            "x": x, "target": tgt, "y_eval": y_eval, "y_train": y_train.detach(),
            "loss": loss.detach(),
            "grads": {k: p.grad.clone() for k, p in model.named_parameters()},
            "buffers_after": {k: b.clone() for k, b in model.named_buffers()},
        }
        fixtures.save(out, HERE, name)
        print(name, "->", HERE, "loss", float(loss))


if __name__ == "__main__":
    main()
