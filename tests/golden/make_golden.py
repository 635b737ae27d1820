"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref, built from
/root/reference by `make -C oracle ref`). Run in the build container only:

    python tests/golden/make_golden.py

Each file holds the input edge list and the reference's [E',3] float64 output for one
(graph, o_v, o_n) with the injected seeds recorded (sample_seed = the reference's default
mt19937_64 seed 5489; rd_seed feeds the stand-in for std::random_device).

    python tests/golden/make_golden.py --ref-build-cases [--from-oracle-ref-mode]

writes tests/golden/ref_build/cases.npz instead: the inputs of the reference-build comparison
(tests/util.py reference_build_cases, seeds REF_BUILD_SEEDS) and, per (case, o_v, o_n), the row count, the SHA-256
of the whole [E',3] float64 output and a seeded sample of its rows. Whole outputs of these larger graphs would be
~1.3 MB. The outputs come from the reference build, or with --from-oracle-ref-mode from the oracle's reference
mode; the file's `source` entry says which.

    python tests/golden/make_golden.py --keyed-cases

writes tests/golden/keyed/cases.npz: for every run of tests/util.py keyed_pin_runs, its id and the SHA-256 of the
keyed oracle's output (row, col and fp32 weight bytes), stats and elimination order (util.keyed_digest). Regenerating
on a later tree must give the same arrays; `source` records the commit the digests were first taken on."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from rlap_b200 import graphs  # noqa: E402
from tests import util  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF_BUILD_PATH = os.path.join(HERE, "ref_build", "cases.npz")
KEYED_PATH = os.path.join(HERE, "keyed", "cases.npz")
SAMPLE_ROWS = 64

# what --from-oracle-ref-mode records as the source: refmode in oracle/rlap_oracle.cc, ref_driver.cc and
# ref_seed_inject.h are unchanged since commit c4ca53b, whose test_ref_mode_matches_reference_build compared this
# mode bit for bit with the reference build on exactly these inputs and seeds
ORACLE_SOURCE = ("oracle reference mode (oracle/rlap_oracle.cc refmode, unchanged since c4ca53b, where it matched the "
                 "reference build bit for bit on these cases)")

KEYED_SOURCE = ("oracle keyed mode at commit 8ecb4b5 (unmasked runs: oracle_keyed_schur; masked runs: the keep-mask "
                "copy of its driver that commit had)")


def sample_index(rows: int) -> np.ndarray:
    return np.sort(np.random.default_rng(rows).choice(rows, min(rows, SAMPLE_ROWS), replace=False))


def main():
    assert ref.available(), "build oracle/_ref first (make -C oracle ref)"
    cases = [("ba100", graphs.barabasi_albert(100, 50, seed=1), 100, 50, None),
             ("ba100w", graphs.barabasi_albert(100, 50, seed=2), 100, 50, "w"),
             ("sbm300", graphs.sbm(300, 4, 900, seed=5), 300, 90, None)]
    for name, ei, n, t, wmode in cases:
        w = util.sym_weights(ei).astype(np.float64) if wmode else None
        info = util.edge_info(ei, w)
        for o_v, o_n in util.COMBOS:
            out = ref.approximate_cholesky(info, n, t, o_v, o_n, sample_seed=5489, rd_seed=17)
            np.savez_compressed(os.path.join(HERE, f"{name}_{o_v}_{o_n}.npz"), edge_info=info, n=n, t=t,
                                sample_seed=5489, rd_seed=17, out=out)
    print("golden vectors written to", HERE)


def ref_build_cases(from_oracle: bool):
    if from_oracle:
        from oracle import port
        run, source = port.ref_approximate_cholesky, ORACLE_SOURCE
    else:
        assert ref.available(), "build oracle/_ref first (make -C oracle ref)"
        run, source = ref.approximate_cholesky, "reference build (oracle/_ref)"
    data = {"source": np.array(source), "sample_seed": util.REF_BUILD_SEEDS["sample_seed"],
            "rd_seed": util.REF_BUILD_SEEDS["rd_seed"]}
    names, count, digest, sidx, sample = [], [], [], [], []
    for name, ei, w, n, t in util.reference_build_cases():
        data[f"{name}_edge_index"] = ei.astype(np.uint16)
        if w is not None:
            data[f"{name}_weights"] = w.astype(np.float32)       # sym_weights is float32: exact
        data[f"{name}_n"], data[f"{name}_t"] = n, t
        info = util.edge_info(ei, w)
        for o_v, o_n in util.COMBOS:
            out = run(info, n, t, o_v, o_n, **util.REF_BUILD_SEEDS)
            idx = sample_index(out.shape[0])
            names.append(f"{name}_{o_v}_{o_n}")
            count.append(out.shape[0])
            digest.append(util.output_digest(out))
            sidx.append(idx)
            sample.append(out[idx])
    data.update(case=np.array(names), count=np.array(count, dtype=np.int64), digest=np.stack(digest),
                sample_index=np.stack(sidx).astype(np.int32), sample=np.stack(sample))
    os.makedirs(os.path.dirname(REF_BUILD_PATH), exist_ok=True)
    np.savez_compressed(REF_BUILD_PATH, **data)
    print("reference-build cases written to", REF_BUILD_PATH, "from", source)


def keyed_cases():
    from oracle import port
    ids, digest = [], []
    for case, ptr, col, w, kw in util.keyed_pin_runs(port):
        ids.append(case)
        digest.append(util.keyed_digest(port, ptr, col, w, kw))
    os.makedirs(os.path.dirname(KEYED_PATH), exist_ok=True)
    np.savez_compressed(KEYED_PATH, source=np.array(KEYED_SOURCE), case=np.array(ids), digest=np.stack(digest))
    print(len(ids), "keyed-mode digests written to", KEYED_PATH)


if __name__ == "__main__":
    if "--ref-build-cases" in sys.argv:
        ref_build_cases("--from-oracle-ref-mode" in sys.argv)
    elif "--keyed-cases" in sys.argv:
        keyed_cases()
    else:
        main()
