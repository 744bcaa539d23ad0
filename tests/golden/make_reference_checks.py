"""Generate the stored results of the reference's own code that the CPU tests compare against:

  reference_checks.npz          - training-mode outputs of the reference's modules (test_cpu_oracle.py),
                                  its `_detect_peaks` picks (test_cpu_postprocess.py) and its `_normalize` /
                                  `_generate_soft_label` results (test_cpu_preprocess.py);
  reference_dropout_sites.json  - every nn.Dropout / DropPath site of the reference models with its rate
                                  (test_cpu_oracle.py).

Run where a checkout of the unmodified reference is present (SEIST_REFERENCE_ROOT, see oracle/reference_import.py):

    python tests/golden/make_reference_checks.py

The inputs are rebuilt by the tests from the same seeds; each input set also stores a strided probe of itself so that
a change in a random stream shows up as such and not as a mismatch of the code under test.
"""
import ast
import json
import os
import sys
from typing import Any, List, Tuple, Union
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)
import reference_inputs as I  # noqa: E402
from oracle import reference_import as ri  # noqa: E402
from oracle import postprocess_ref as PR  # noqa: E402


def _reference_source_functions(rel_path, top_level=(), methods_of=None, methods=()):
    """Functions of one reference module, executed from their source (the modules themselves import h5py / obspy /
    pandas-backed code that is not needed by these functions)."""
    path = os.path.join(ri.REF_ROOT, rel_path)
    tree = ast.parse(open(path).read())
    ns = {"np": np, "Tuple": Tuple, "Union": Union, "List": List, "Any": Any}
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in top_level]
    if methods_of:
        cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == methods_of)
        body += [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in methods]
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)      # noqa: S102 - the reference's own code
    return ns


def module_outputs(M, out):
    for name in I.MODULE_MODELS:
        sd, x = I.module_inputs(name)
        ref = ri.zero_drop_rates(M.create_model(name, in_channels=3, in_samples=I.MODULE_L))
        ref.load_state_dict(sd, strict=True)
        ref.train()
        with torch.no_grad():
            out[f"modules.{name}.y"] = ref(x).numpy()
        out[f"modules.{name}.x_probe"] = I.probe(x.numpy())


def dropout_sites(M):
    sites = {}
    for name in I.DROPOUT_MODELS:
        ref = M.create_model(name, in_channels=3, in_samples=1024)
        rows = []
        for path, mod in ref.named_modules():
            cls = mod.__class__.__name__
            if cls == "Dropout":
                rows.append([path, float(mod.p)])
            elif cls == "DropPath":
                rows.append([path, float(mod.drop_prob or 0.0)])
        sites[name] = rows
    return sites


def picks(out):
    detect_peaks = _reference_source_functions("training/postprocess.py", top_level=("_detect_peaks",))["_detect_peaks"]
    for topk, mpd in I.PICK_CASES:
        x = I.pick_traces(topk, mpd)
        out[f"pick.{topk}_{mpd}.x_probe"] = I.probe(x)
        for thr in I.PICK_THRESHOLDS:
            want = np.full((x.shape[0], topk), PR.PAD_PHASE, dtype=np.int64)
            for i, row in enumerate(x):
                p = detect_peaks(row, mph=thr, mpd=mpd, topk=topk)
                want[i, :p.size] = p
            out[f"pick.{topk}_{mpd}.{thr}"] = want


def preprocess(out):
    ns = _reference_source_functions("training/preprocess.py", top_level=("_pad_phases",), methods_of="DataPreprocessor",
                                     methods=("_normalize", "_generate_soft_label"))
    for mode, x in I.normalize_inputs():
        out[f"normalize.{mode or 'none'}"] = ns["_normalize"](None, x.copy(), mode)
    me = SimpleNamespace(coda_ratio=I.CODA_RATIO, dtype=np.float32, data_channels=["z", "n", "e"])
    for shape, width, ci, ppks, spks in I.label_cases():
        ev = {"data": np.zeros((3, I.LABEL_L), np.float32), "ppks": list(ppks), "spks": list(spks)}
        out[f"labels.{shape}.{width}.{ci}"] = np.stack(
            [ns["_generate_soft_label"](me, row, ev, width, shape) for row in ("det", "ppk", "spk")])


def main():
    M = ri.import_reference_models()
    out = {}
    module_outputs(M, out)
    picks(out)
    preprocess(out)
    np.savez_compressed(os.path.join(HERE, "reference_checks.npz"), **out)
    with open(os.path.join(HERE, "reference_dropout_sites.json"), "w") as f:
        json.dump(dropout_sites(M), f, indent=0)
        f.write("\n")
    for fn in ("reference_checks.npz", "reference_dropout_sites.json"):
        print(fn, os.path.getsize(os.path.join(HERE, fn)) // 1024, "KiB")


if __name__ == "__main__":
    main()
