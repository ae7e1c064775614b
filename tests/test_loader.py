"""CPU: gnn_rag_b200.loader.build_fact_mat is a bit-identical drop-in for the reference's
BasicDataLoader._build_fact_mat (gnn/dataset_load.py:473-527) -- against golden outputs of the unmodified reference
(tests/golden/loader/fact_mat_*.npz, made by tests/golden/make_fact_mat_golden.py), including larger random loader
states (with a timing comparison)."""
import os
import time

import numpy as np
import pytest

from gnn_rag_b200 import loader
from loader_fixture import CASES, LARGE_CASES, FakeLoader

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loader")
KEYS = ("heads", "rels", "tails", "batch_ids", "fact_ids", "weight_list", "weight_rel_list")


def assert_same(got, want):
    for k, g, w in zip(KEYS, got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, k
        assert g.dtype.kind == w.dtype.kind, k
        assert np.array_equal(g, w), k           # bit-identical, floats included


@pytest.mark.parametrize("name", sorted(CASES))
def test_build_fact_mat_matches_reference_golden(name):
    kw, ids, dropout, seed = CASES[name]
    gold = np.load(os.path.join(GOLD, "fact_mat_%s.npz" % name))
    np.random.seed(seed)
    got = loader.build_fact_mat(FakeLoader(**kw), ids, dropout)
    assert isinstance(got[5], list) and isinstance(got[6], list)        # reference types
    assert got[0].dtype == np.int64
    assert_same(got, [gold[k] for k in KEYS])
    # the RNG stream was consumed exactly like the reference does: the next draw agrees
    np.random.seed(seed)
    for sid in ids:
        np.random.permutation(len(FakeLoader(**kw).kb_adj_mats[sid][0]))
    expect_next = np.random.rand()
    np.random.seed(seed)
    loader.build_fact_mat(FakeLoader(**kw), ids, dropout)
    assert np.random.rand() == expect_next


@pytest.mark.parametrize("name", sorted(CASES))
def test_loader_oracle_matches_reference_golden(name):
    """oracle/loader_oracle.py (the reference-form restatement bench.py times as the CPU get_batch cost) against the
    arrays recorded from the unmodified reference."""
    from oracle import loader_oracle
    kw, ids, dropout, seed = CASES[name]
    gold = np.load(os.path.join(GOLD, "fact_mat_%s.npz" % name))
    np.random.seed(seed)
    got = loader_oracle.build_fact_mat(FakeLoader(**kw), ids, dropout)
    assert_same(got, [gold[k] for k in KEYS])


def test_loader_oracle_state_from_synthetic_batch_round_trip():
    from gnn_rag_b200 import synthetic as S
    from oracle import loader_oracle
    b = S.make_batch(5, B=4, N=30, E=90, num_entity=500, num_relation=12, num_word=50, n_real="ragged")
    st = loader_oracle.state_from_batch(b, 12)
    np.random.seed(0)
    got = loader_oracle.build_fact_mat(st, list(range(4)), 0.0)
    key = lambda h, r, t: sorted(zip(h.tolist(), r.tolist(), t.tolist()))          # same multiset of facts
    assert key(got[0], got[1], got[2]) == key(b[2][0], b[2][1], b[2][2])


def test_variants_and_install():
    kw, ids, dropout, seed = CASES["small"]
    ld = FakeLoader(**kw)
    np.random.seed(seed)
    base = loader.build_fact_mat(ld, ids, dropout)
    np.random.seed(seed)
    arr = loader.build_fact_mat(ld, ids, dropout, weights="arrays", index_dtype=np.int32)
    assert arr[0].dtype == np.int32 and isinstance(arr[5], np.ndarray) and arr[5].dtype == np.float64
    assert_same([a.astype(np.int64) if a.dtype == np.int32 else a for a in arr], base)
    np.random.seed(seed)
    none = loader.build_fact_mat(ld, ids, dropout, weights="none")
    assert none[5] is None and none[6] is None and np.array_equal(none[0], base[0])
    with pytest.raises(ValueError):
        loader.build_fact_mat(ld, ids, dropout, weights="bogus")

    class L(FakeLoader):
        def _build_fact_mat(self, sample_ids, fact_dropout):
            raise AssertionError("not patched")

    orig = loader.install(L, weights="arrays")
    try:
        np.random.seed(seed)
        assert_same(L(**kw)._build_fact_mat(ids, dropout), base)
    finally:
        L._build_fact_mat = orig
    inst = L(**kw)
    loader.install(inst)
    np.random.seed(seed)
    assert_same(inst._build_fact_mat(ids, dropout), base)


def test_unshuffled_offset_concat_is_the_same_batch_up_to_fact_order():
    """shuffle=False (serving, SURVEY 8f row 3): per question the same multiset of facts with the same weights, stored
    order, RNG untouched."""
    kw, ids, _dropout, seed = CASES["small"]
    ld = FakeLoader(**kw)
    np.random.seed(seed)
    want = loader.build_fact_mat(ld, ids, 0.0, weights="arrays")
    np.random.seed(seed)
    state = np.random.get_state()[1].copy()
    got = loader.build_fact_mat(ld, ids, 0.0, weights="arrays", shuffle=False)
    assert np.array_equal(np.random.get_state()[1], state)             # no RNG draw
    assert hasattr(ld, "_gr_flat")
    assert np.array_equal(got[3], want[3]) and np.array_equal(got[4], want[4])

    def rows(t):
        return sorted(zip(t[3].tolist(), t[0].tolist(), t[1].tolist(), t[2].tolist(), t[5].tolist(), t[6].tolist()))
    assert rows(got) == rows(want)
    h, r, t = ld.kb_adj_mats[ids[0]]                                   # first question keeps its stored order
    assert np.array_equal(got[0][: len(h)], h) and np.array_equal(got[1][: len(h)], r)
    i32 = loader.build_fact_mat(ld, ids, 0.0, weights="none", index_dtype=np.int32, shuffle=False)
    assert i32[0].dtype == np.int32 and np.array_equal(i32[0], got[0])
    with pytest.raises(ValueError):
        loader.build_fact_mat(ld, ids, 0.2, shuffle=False)


def test_build_fact_mat_matches_reference_golden_large_and_is_faster():
    """Larger loader states: bit-identical to the reference's output (golden), and faster than the reference-form
    restatement (oracle/loader_oracle.py), which is checked against the same golden."""
    from oracle import loader_oracle
    for name in sorted(LARGE_CASES):
        kw, ids, dropout, seed = LARGE_CASES[name]
        want = np.load(os.path.join(GOLD, "fact_mat_%s.npz" % name))
        want = [want[k] for k in KEYS]
        ld = FakeLoader(**kw)
        np.random.seed(seed)
        t0 = time.perf_counter()
        ref_form = loader_oracle.build_fact_mat(ld, ids, dropout)
        t_ref = time.perf_counter() - t0
        np.random.seed(seed)
        t0 = time.perf_counter()
        got = loader.build_fact_mat(ld, ids, dropout)
        t_new = time.perf_counter() - t0
        assert got[0].dtype == np.int64
        assert_same(got, want)
        assert_same(ref_form, want)
        assert t_new < t_ref, (name, t_new, t_ref)
