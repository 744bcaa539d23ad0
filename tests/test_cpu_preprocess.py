"""not-gpu: the input-side oracle (oracle/preprocess_ref.py) against the results of the reference's own `_normalize`,
`_pad_phases` and `_generate_soft_label`, stored in tests/golden/reference_checks.npz
(tests/golden/make_reference_checks.py)."""
import os

import numpy as np

import reference_inputs as I
from oracle import preprocess_ref as PR

REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))


def test_input_side_oracle_matches_reference_sources():
    for mode, x in I.normalize_inputs():
        want = REF[f"normalize.{mode or 'none'}"]
        assert np.array_equal(PR.normalize(x, mode), want), mode
    for shape, width, ci, ppks, spks in I.label_cases():
        got = PR.dpk_labels(ppks, spks, I.LABEL_L, width, shape, I.CODA_RATIO)
        want = REF[f"labels.{shape}.{width}.{ci}"]
        for row, name in enumerate(("det", "ppk", "spk")):
            assert np.array_equal(got[row], want[row]), (shape, width, ppks, spks, name)
