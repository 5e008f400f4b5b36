"""CPU: the oracle restatement against the reference's own known-answer tests (pins the oracle)."""
import numpy as np
import pytest

import oracle
from oracle import sort as osort
from tests.golden import sort_cases as G
from tests.helpers import ALL_DTYPES, make_col

TYPED = [np.int8, np.int16, np.int32, np.int64, np.uint8, np.uint16, np.uint32, np.uint64, np.float32, np.float64]


@pytest.mark.parametrize("case", G.SORTED_ORDER_CASES, ids=lambda c: c["name"])
@pytest.mark.parametrize("dtype", TYPED + [np.bool_])
def test_sorted_order_golden(case, dtype):
    if dtype == np.bool_ and case["skip_bool"]:
        pytest.skip("the reference does not pin bool order for this case")
    cols = [make_col(v, dtype if k == "T" else np.int32) for v, k in case["cols"]]
    got = osort.sorted_order(cols, case["order"], case["nulls"])
    assert got.tolist() == case["expected"], case["cite"]


@pytest.mark.parametrize("dtype", TYPED)
def test_sliced_columns(dtype):
    c1 = make_col(G.SLICED["col1"], np.int32)
    c2 = make_col(G.SLICED["col2"], dtype)
    assert osort.sorted_order([c1, c2], [0, 0]).tolist() == G.SLICED["expected"]
    k = G.SLICED["split"]
    s1 = (c1[0][k:], c1[1][k:])
    assert osort.sorted_order([s1, s1], [0, 0]).tolist() == G.SLICED["expected_sliced"]


@pytest.mark.parametrize("dtype", TYPED)
def test_single_column(dtype):
    for case, valid in ((G.SINGLE_NO_NULL, None), (G.SINGLE_WITH_NULL, G.SINGLE_WITH_NULL["valid"])):
        vals = [v if (valid is None or valid[i]) else None for i, v in enumerate(case["values"])]
        col = make_col(vals, dtype)
        exp = case["expected_unsigned"] if np.dtype(dtype).kind == "u" else case["expected_signed"]
        got = osort.sorted_order([col], [0], [1])
        # the reference compares gathered values (run_stable_sort_test), not indices
        gv = osort.gather([col], got)[0]
        ev = osort.gather([col], exp)[0]
        gm = np.ones(len(got), bool) if gv[1] is None else gv[1]
        em = np.ones(len(got), bool) if ev[1] is None else ev[1]
        assert np.array_equal(gm, em)
        assert np.array_equal(gv[0][gm], ev[0][em])
        if valid is None:
            assert got.tolist() == exp  # no ties among nulls: a stable order is unique


def test_inf_nan():
    col = (np.array(G.INF_NAN["values"], dtype=np.float64), None)
    assert osort.sorted_order([col]).tolist() == G.INF_NAN["expected"]
    # descending (not pinned by the reference): tuple (isnan*(idx+1), f) sorted descending
    got = osort.sorted_order([col], [1]).tolist()
    assert got[:6] == [13, 12, 9, 3, 2, 1]
    assert got[6:] == [4, 10, 6, 8, 7, 0, 14, 5, 11]


def test_size_mismatch_throws():
    # sort_test.cpp:667-698 MismatchInColumnOrderSize / MismatchInNullPrecedenceSize
    c = make_col([1, 2, 3], np.int32)
    with pytest.raises(RuntimeError):
        osort.sorted_order([c, c], [0])
    with pytest.raises(RuntimeError):
        osort.sorted_order([c, c], [0, 0], [1])
    # sort_test.cpp:962-978 sort_by_key size mismatch
    with pytest.raises(RuntimeError):
        osort.sort_by_key([make_col([1, 2], np.int32)], [c])
    # sort_test.cpp:700-717 zero sized
    assert len(osort.sorted_order([(np.empty(0, np.int32), None)])) == 0


def test_join_gold_maps():
    # join_tests.cpp:2316-2337 (gold maps) with the InnerJoinNoNulls column 0 (:1163-1237)
    l, r = oracle.join.inner_join([(np.array([3, 1, 2, 0, 2]), None)], [(np.array([2, 2, 0, 4, 3]), None)])
    assert l.tolist() == [0, 2, 2, 3, 4, 4] and r.tolist() == [4, 0, 1, 2, 0, 1]


def test_murmur3_row_hash_pinned():
    """oracle/partition.py: MurmurHash3_x86_32 against the published known answers (SMHasher verification values) and against
    scikit-learn's C implementation on random fixed-width values (tests/golden/murmur3_sklearn.npz: 300 values per dtype and
    murmurhash3_32(value bytes, seed, positive=True) for seeds 0 and 619, computed with scikit-learn 1.9.0); hash_combine and the
    null hash against hand-computed values (cpp/include/cudf/hashing/detail/hashing.hpp:83-86, row_operator/hashing.cuh:52-56)."""
    from pathlib import Path

    import numpy as np

    from oracle import partition as op

    known = [(np.uint32, 0xFFFFFFFF, 0, 0x76293B50), (np.uint32, 0x87654321, 0, 0xF55B516B), (np.uint32, 0x87654321, 0x5082EDEE, 0x2362F9DE),
             (np.uint16, 0x4321, 0, 0xA0F7B07A), (np.uint8, 0x21, 0, 0x72661CF4), (np.uint32, 0, 0, 0x2362F9DE)]
    for dt, v, seed, exp in known:
        assert int(op.murmur3_32_fixed(np.array([v], dt), seed)[0]) == exp
    gold = np.load(Path(__file__).resolve().parent / "golden" / "murmur3_sklearn.npz")
    for dt in (np.uint8, np.uint16, np.uint32, np.uint64, np.float32, np.float64):
        v = gold[f"{np.dtype(dt).name}_values"]
        assert v.dtype == dt and len(v) == 300
        for seed in (0, 619):
            assert np.array_equal(op.murmur3_32_fixed(v, seed), gold[f"{np.dtype(dt).name}_seed{seed}"])
    # normalisation and nulls: -0.0 hashes like +0.0, every NaN like the canonical one, a null is UINT32_MAX
    f = np.array([0.0, -0.0, np.nan, -np.nan], np.float64)
    h = op.row_hash([(f, np.array([True, True, True, True]))])
    assert h[0] == h[1] and h[2] == h[3]
    assert int(op.row_hash([(f, np.array([False, True, True, True]))])[0]) == 0xFFFFFFFF
    a = np.array([1, 2], np.int32)
    h0, h1 = op.murmur3_32_fixed(a), op.murmur3_32_fixed(a.astype(np.int64))
    comb = h0 ^ ((h1 + np.uint32(0x9E3779B9) + (h0 << np.uint32(6)) + (h0 >> np.uint32(2))).astype(np.uint32))
    assert np.array_equal(op.row_hash([(a, None), (a.astype(np.int64), None)]), comb)


def test_mix64_shuffle_bucket_pinned():
    """oracle/partition.py::mix64 is MurmurHash3's fmix64: fixed point 0, the widely quoted fmix64(1) = 0xB456BCFC34C2CB2C, and
    agreement with an independent big-integer restatement; shuffle_bucket stays inside [0, P) and is balanced."""
    import numpy as np

    from oracle import partition as op

    M = (1 << 64) - 1

    def fmix(k):
        k ^= k >> 33; k = k * 0xFF51AFD7ED558CCD & M
        k ^= k >> 33; k = k * 0xC4CEB9FE1A85EC53 & M
        return k ^ (k >> 33)

    assert int(op.mix64(np.array([0], np.uint64))[0]) == 0
    assert int(op.mix64(np.array([1], np.uint64))[0]) == 0xB456BCFC34C2CB2C
    rng = np.random.default_rng(3)
    v = rng.integers(0, 2**64 - 1, 500, dtype=np.uint64)
    assert [int(x) for x in op.mix64(v)] == [fmix(int(x)) for x in v]
    k = rng.integers(-2**63, 2**63 - 1, 200_000, dtype=np.int64)
    for P in (2, 3, 8):
        b = op.shuffle_bucket(k, P)
        assert b.min() >= 0 and b.max() < P
        assert np.abs(np.bincount(b, minlength=P) / len(k) - 1 / P).max() < 0.01
        assert b[0] == (((fmix(((int(k[0]) & M) ^ (1 << 63)) + 0x9E3779B97F4A7C15 & M) >> 32) * P) >> 32)
