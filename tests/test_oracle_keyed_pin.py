"""Pins the keyed oracle (oracle/rlap_oracle.cc keyed mode, the specification of the CUDA path) to stored digests: for
every run of util.keyed_pin_runs - all modes, unit and hashed weights, with and without a keep mask, both removal
counts, a non-zero view, a shared order and full-clique mode - the SHA-256 of its output rows (row, col, fp32 weight),
its stats and its elimination order equals the one in tests/golden/keyed/cases.npz
(tests/golden/make_golden.py --keyed-cases; `source` in the file says which commit the digests were taken on)."""
import os

import numpy as np

from tests import util

KEYED_GOLD = os.path.join(os.path.dirname(__file__), "golden", "keyed", "cases.npz")


def test_keyed_mode_matches_stored_digests(oracle_port):
    z = np.load(KEYED_GOLD)
    ids, bad = [], []
    for case, ptr, col, w, kw in util.keyed_pin_runs(oracle_port):
        k = len(ids)
        ids.append(case)
        if k < z["case"].shape[0] and not np.array_equal(util.keyed_digest(oracle_port, ptr, col, w, kw), z["digest"][k]):
            bad.append(case)
    assert ids == z["case"].tolist()                                       # every stored run, in the stored order
    assert not bad, f"{len(bad)} of {len(ids)} keyed runs differ from their stored digest, first: {bad[:10]}"
