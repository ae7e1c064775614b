"""Golden outputs of the UNMODIFIED reference ``BasicDataLoader._build_fact_mat`` (gnn/dataset_load.py:473-527) on
the stand-in loader states of tests/loader_fixture.py.  Needs a checkout of the original project where
oracle/ref_harness.py looks for it:
    python tests/golden/make_fact_mat_golden.py
writes tests/golden/loader/fact_mat_<case>.npz.  The large cases are stored compressed, with the index arrays narrowed
to int16 (every value fits; the test checks the int64 dtype of the result separately)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from loader_fixture import CASES, LARGE_CASES, FakeLoader  # noqa: E402
from oracle import ref_harness  # noqa: E402


def reference_build_fact_mat():
    ref_harness._import_reference()
    import dataset_load  # noqa: E402  (reference module, imported read-only)
    return dataset_load.BasicDataLoader._build_fact_mat


if __name__ == "__main__":
    fn = reference_build_fact_mat()
    for name, (kw, ids, dropout, seed) in dict(CASES, **LARGE_CASES).items():
        ld = FakeLoader(**kw)
        np.random.seed(seed)
        h, r, t, b, f, w, wr = fn(ld, ids, dropout)
        w, wr = np.asarray(w, dtype=np.float64), np.asarray(wr, dtype=np.float64)
        path = os.path.join(HERE, "loader", "fact_mat_%s.npz" % name)
        if name in LARGE_CASES:
            idx = [h, r, t, b, f]
            assert all(np.array_equal(x.astype(np.int16), x) for x in idx)
            h, r, t, b, f = [x.astype(np.int16) for x in idx]
            np.savez_compressed(path, heads=h, rels=r, tails=t, batch_ids=b, fact_ids=f, weight_list=w,
                                weight_rel_list=wr)
        else:
            np.savez(path, heads=h, rels=r, tails=t, batch_ids=b, fact_ids=f, weight_list=w, weight_rel_list=wr)
        print(name, len(h), "facts")
