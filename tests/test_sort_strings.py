"""SortIndices / select_k_unstable on utf8, large_utf8, binary and large_binary keys (csrc/sort_strings.cu;
ArrayCompareSorter over base-binary types, kernels/vector_array_sort.cc:144-178,588-594).

The order is unsigned byte-wise lexicographic with a proper prefix first; the sort is stable, nulls are partitioned
at_start / at_end, and descending keeps ties in ascending row order.  A restatement of that rule on Python `bytes`
(`string_sort_indices` below) is pinned against the reference binary on CPU; the CUDA path is checked against both on
the GPU, with each internal path forced through B2_SORT_STRINGS_PATH and with the automatic choice."""
import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

from oracle import arrow_oracle as ora
from tests.util import SEED

STRING_TYPES = [pa.utf8(), pa.large_utf8(), pa.binary(), pa.large_binary()]
ORDERS = ["ascending", "descending"]
PLACEMENTS = ["at_end", "at_start"]


# ---- restatement --------------------------------------------------------------------------------------------------
def _as_bytes(v):
    return v.encode() if isinstance(v, str) else v


def string_sort_indices(arr: pa.Array, order="ascending", null_placement="at_end") -> pa.Array:
    """stable sort of the non-null values as Python bytes (unsigned, a proper prefix first), nulls partitioned"""
    vals = [_as_bytes(v) for v in arr.to_pylist()]
    valid = [i for i, v in enumerate(vals) if v is not None]
    nulls = [i for i, v in enumerate(vals) if v is None]
    rest = sorted(valid, key=lambda i: vals[i], reverse=order == "descending")  # reverse=True stays stable
    return pa.array(rest + nulls if null_placement == "at_end" else nulls + rest, pa.uint64())


def sort_indices_multi(cols, keys, null_placement="at_end") -> pa.Array:
    """least-significant key first, as the oracle's numeric multi-key sort; string keys use the restatement above"""
    n = len(next(iter(cols.values())))
    perm = np.arange(n, dtype=np.uint64)
    for name, order in reversed(list(keys)):
        col = cols[name].take(pa.array(perm))
        one = string_sort_indices if _is_string(col.type) else ora.sort_indices
        perm = perm[one(col, order, null_placement).to_numpy().astype(np.int64)]
    return pa.array(perm, pa.uint64())


def _is_string(t):
    return any(t == s for s in STRING_TYPES)


# ---- cases --------------------------------------------------------------------------------------------------------
def _random_strings(n, seed, alphabet="ab\x00é", max_len=20, null_p=0.1):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        if rng.random() < null_p:
            out.append(None)
        else:
            out.append("".join(alphabet[j] for j in rng.integers(0, len(alphabet), rng.integers(0, max_len + 1))))
    return out


_P = "x" * 300
CASES = {
    "empty": [],
    "one": ["x"],
    "one_null": [None],
    "all_null": [None] * 5,
    "empty_strings": ["", None, "", "a", "", None, "\x00"],
    "nul_suffix": ["ab\x00", "ab", "a", "ab", "ab\x00\x00", "b", "ab\x00", "aa\xff"[:2]],
    "lengths": [s for L in (15, 14, 8, 7, 6) for s in ("abcdefghijklmno"[:L], "abcdefghijklmnz"[:L - 1] + "z")] * 2,
    "high_bytes": ["é", "e", "z", "ÿ", "\u0080", "A", "é", "ée", "￿", "\U0001f600", "~"],
    "prefix_300": [_P + "b", _P, _P + "a", _P + "aq", _P[:-1] + "y", _P + "b", None, _P + "a", _P[:150]],
    "random": _random_strings(3000, SEED),
    "few_distinct": _random_strings(3000, SEED + 1, alphabet="ab", max_len=3),
}
BINARY_ONLY = {"raw_bytes": [b"\xff", b"\x80", b"\x7f", b"\x00", b"", b"\xff\x00", b"\xff", None, b"\x80\x80"]}


def make(values, t, pad=3):
    """the case as an array of type t, sliced so that its offsets and validity start at a non-zero position"""
    head = ["pad"] * pad
    if pa.types.is_binary(t) or pa.types.is_large_binary(t):
        full = pa.array([_as_bytes(v) for v in head + values], t)
    else:
        full = pa.array(head + values, t)
    return full.slice(pad)


def all_cases():
    for t in STRING_TYPES:
        for name, vals in CASES.items():
            yield f"{t}-{name}", make(vals, t)
        if pa.types.is_binary(t) or pa.types.is_large_binary(t):
            for name, vals in BINARY_ONLY.items():
                yield f"{t}-{name}", make(vals, t)


def reference(arr, order, placement):
    return pc.array_sort_indices(arr, order=order, null_placement=placement)


# ---- CPU: the restatement against the reference binary --------------------------------------------------------------
@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("order", ORDERS)
def test_restatement_matches_the_reference_binary(order, placement):
    for name, arr in all_cases():
        assert string_sort_indices(arr, order, placement).equals(reference(arr, order, placement)), name


def mixed_table(n, seed=SEED):
    rng = np.random.default_rng(seed)
    words = np.array(["", "a", "ab", "ab\x00", "b", "é", "abcdefgh", "abcdefghi"], dtype=object)
    s = words[rng.integers(0, len(words), n)]
    t = [bytes(rng.integers(0, 3, rng.integers(0, 10)).astype(np.uint8)) for _ in range(n)]
    return {
        "s": pa.array(list(s), pa.utf8(), mask=rng.random(n) < 0.1),
        "t": pa.array(t, pa.large_binary(), mask=rng.random(n) < 0.1),
        "i": pa.array(rng.integers(0, 4, n).astype(np.int32), mask=rng.random(n) < 0.1),
        "f": pa.array(rng.integers(0, 3, n).astype(np.float64)),
    }


MIXED_KEYS = [
    [("s", "ascending"), ("i", "descending")],           # string first
    [("i", "ascending"), ("f", "descending"), ("s", "descending")],  # string last
    [("s", "descending"), ("t", "ascending")],           # two string keys
    [("t", "descending"), ("i", "ascending"), ("s", "ascending")],
]


@pytest.mark.parametrize("placement", PLACEMENTS)
def test_multi_key_restatement_matches_the_reference_binary(placement):
    for n in (0, 1, 2, 700):
        cols = mixed_table(n)
        for keys in MIXED_KEYS:
            want = pc.sort_indices(pa.table(cols), sort_keys=keys, null_placement=placement)
            assert sort_indices_multi(cols, keys, placement).equals(want), (n, keys)


@pytest.mark.parametrize("order", ORDERS)
def test_select_k_restatement_matches_the_reference_binary(order):
    for t in STRING_TYPES:
        arr = make(_random_strings(3000, SEED + 2), t)
        for k in (1, 10, 500):
            got = string_sort_indices(arr, order).slice(0, k)
            want = pc.select_k_unstable(arr, k, sort_keys=[("x", order)])
            assert pc.take(arr, got).equals(pc.take(arr, want)), (t, k)


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(params=[None, "dict", "refine"], ids=["auto", "dict", "refine"])
def path(request, monkeypatch):
    if request.param is None:
        monkeypatch.delenv("B2_SORT_STRINGS_PATH", raising=False)
    else:
        monkeypatch.setenv("B2_SORT_STRINGS_PATH", request.param)
    return request.param


def _dev(arr, ctx):
    from arrow_b200 import DeviceArray
    return DeviceArray.from_arrow(arr, ctx)


@pytest.mark.gpu
def test_gpu_sort_matches_restatement_and_reference(ctx, path):
    import arrow_b200.compute as bc
    cases = list(all_cases())
    # large enough for the automatic choice to sample: many duplicates (dictionary side) and all distinct (refinement)
    rng = np.random.default_rng(SEED + 3)
    words = [f"w{j:05d}-{'q' * (j % 11)}" for j in range(2000)]
    dup = [words[j] for j in rng.integers(0, len(words), 300_000)]
    uniq = [f"{j * 7919 % 300_001:09d}" for j in range(300_000)]
    for t in (pa.utf8(), pa.large_binary()):
        cases.append((f"{t}-dup300k", make(dup, t)))
        cases.append((f"{t}-unique300k", make(uniq, t)))
    for name, arr in cases:
        d = _dev(arr, ctx)
        for order in ORDERS:
            for placement in PLACEMENTS:
                got = bc.array_sort_indices(d, order, placement).to_arrow()
                want = reference(arr, order, placement)
                assert got.equals(want), (path, name, order, placement)
                if len(arr) <= 3000:
                    assert got.equals(string_sort_indices(arr, order, placement)), (path, name, order, placement)


@pytest.mark.gpu
def test_gpu_sort_payload_on_strings(ctx, path):
    import arrow_b200.compute as bc
    rng = np.random.default_rng(SEED + 4)
    arr = make(_random_strings(50_000, SEED + 5, max_len=12), pa.large_utf8())
    payload = pa.array(rng.permutation(len(arr)).astype(np.uint32))
    for order in ORDERS:
        for placement in PLACEMENTS:
            got = bc.sort_payload(_dev(arr, ctx), _dev(payload, ctx), order, placement).to_arrow()
            want = payload.take(reference(arr, order, placement)).cast(pa.uint64())
            assert got.equals(want), (path, order, placement)


@pytest.mark.gpu
@pytest.mark.parametrize("placement", PLACEMENTS)
def test_gpu_multi_key_with_string_keys(ctx, placement, path):
    import arrow_b200.compute as bc
    for n in (0, 1, 700):
        cols = mixed_table(n)
        dcols = {k: _dev(v, ctx) for k, v in cols.items()}
        for keys in MIXED_KEYS:
            got = bc.sort_indices(dcols, sort_keys=keys, null_placement=placement).to_arrow()
            assert got.equals(pc.sort_indices(pa.table(cols), sort_keys=keys, null_placement=placement)), (n, keys)
    n = 2_000_003
    cols = {k: v.slice(3) for k, v in mixed_table(n, SEED + 6).items()}  # non-zero offsets on every key
    dcols = {k: _dev(v, ctx) for k, v in cols.items()}
    for keys in MIXED_KEYS[:3]:
        got = bc.sort_indices(dcols, sort_keys=keys, null_placement=placement).to_arrow()
        assert got.equals(pc.sort_indices(pa.table(cols), sort_keys=keys, null_placement=placement)), keys


def _words(n, distinct, seed, lo=8, hi=16):
    """n large_utf8 values drawn from `distinct` random words of lo..hi bytes (letters)"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi + 1, distinct)
    offs = np.zeros(distinct + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    chars = rng.integers(97, 123, int(offs[-1]), dtype=np.uint8)
    vocab = pa.LargeStringArray.from_buffers(distinct, pa.py_buffer(offs), pa.py_buffer(chars))
    return vocab.take(pa.array(rng.integers(0, distinct, n)))


@pytest.mark.gpu
def test_gpu_select_k_strings(ctx):
    import arrow_b200.compute as bc
    n = 2_000_000
    for name, arr in (("ties", _words(n, 5000, SEED + 7, 1, 9)), ("distinct", _words(n, 1_500_000, SEED + 8))):
        arr = pa.array(arr.to_pylist(), pa.utf8(), mask=np.random.default_rng(SEED).random(n) < 0.05).slice(2)
        d = _dev(arr, ctx)
        m = len(arr)
        for order in ORDERS:
            for placement in PLACEMENTS:
                full = bc.array_sort_indices(d, order, placement).to_arrow()
                assert full.equals(reference(arr, order, placement)), (name, order, placement)
                for k in (0, 1, 37, 1001, 20_000, m // 8, m // 8 + 1, m, m + 5):
                    got = bc.select_k_unstable(d, k, [("x", order)], null_placement=placement).to_arrow()
                    assert got.equals(full.slice(0, min(k, m))), (name, order, placement, k)
        # ties straddling the threshold: the k-th value repeats before and after position k
        full = bc.array_sort_indices(d).to_arrow().to_numpy()
        vals = arr.take(pa.array(full[:30_000])).to_pylist()
        k = next(j for j in range(1000, 29_000) if vals[j - 1] == vals[j] == vals[j - 2])
        got = bc.select_k_unstable(d, k, [("x", "ascending")]).to_arrow()
        assert got.to_numpy().tolist() == full[:k].tolist(), (name, k)
        want = pc.select_k_unstable(arr, k, sort_keys=[("x", "ascending")])
        assert pc.take(arr, got).equals(pc.take(arr, want)), name


@pytest.mark.gpu
def test_gpu_sort_20m_rows(ctx, path):
    import arrow_b200.compute as bc
    n = 20_000_000
    rng = np.random.default_rng(SEED + 9)
    words = _words(n, 1_000_000, SEED + 10)
    lens = rng.integers(8, 33, n)
    offs = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    distinct = pa.LargeStringArray.from_buffers(n, pa.py_buffer(offs), pa.py_buffer(rng.integers(32, 127, int(offs[-1]), dtype=np.uint8)))
    for name, arr in (("1M words", words), ("all distinct", distinct)):
        d = _dev(arr, ctx)
        for order in ORDERS:
            got = bc.array_sort_indices(d, order).to_arrow()
            assert got.equals(reference(arr, order, "at_end")), (path, name, order)


@pytest.mark.gpu
def test_gpu_automatic_path_choice(ctx, monkeypatch):
    """the sample estimates rows per distinct value of the whole column, not of the sample"""
    import arrow_b200.compute as bc
    monkeypatch.delenv("B2_SORT_STRINGS_PATH", raising=False)
    n = 20_000_000
    rng = np.random.default_rng(SEED + 12)
    words = _words(n, 1_000_000, SEED + 13)  # 20 rows per word; a 64Ki sample sees most words once
    assert bc.sort_strings_path(_dev(words, ctx)) == "dict"
    uniq = pa.array([f"{j:012d}" for j in rng.permutation(2_000_000)], pa.large_utf8())
    assert bc.sort_strings_path(_dev(uniq, ctx)) == "refine"
    # 90 % nulls over distinct values: the nulls must not count as one heavily repeated value
    mostly_null = pa.array(uniq.to_pylist(), pa.large_utf8(), mask=rng.random(len(uniq)) < 0.9)
    assert bc.sort_strings_path(_dev(mostly_null, ctx)) == "refine"
    assert bc.sort_strings_path(_dev(make(CASES["random"], pa.utf8()), ctx)) == "refine"  # small columns: no sample
    monkeypatch.setenv("B2_SORT_STRINGS_PATH", "dict")
    assert bc.sort_strings_path(_dev(uniq, ctx)) == "dict"


@pytest.mark.gpu
def test_gpu_cpp_plugin_parity():
    """the C++ drop-in (arrow_b200/cpp/b200_sort_strings_test.cc): array_sort_indices, sort_indices on a device record
    batch, select_k_unstable and b200_order_by with string keys equal the stock registry / order_by node"""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "arrow_b200", "lib", "b200_sort_strings_test")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    tail = "\n".join(p.stdout.splitlines()[-15:])
    assert p.returncode == 0, tail + p.stderr[-2000:]
    assert "PASS" in p.stdout and "FAIL" not in p.stdout, tail


@pytest.mark.gpu
def test_gpu_sort_more_than_4gib_of_characters(ctx):
    """offsets past 2^32: 36M values of 120 bytes whose first 16 bytes are 'a' / 'b' (three rounds), the rest random"""
    import arrow_b200.compute as bc
    n, w = 36_000_000, 120
    rng = np.random.default_rng(SEED + 11)
    chars = rng.integers(0, 256, (n, w), dtype=np.uint8)
    chars[:, :16] = 97 + rng.integers(0, 2, (n, 16), dtype=np.uint8)
    offs = np.arange(n + 1, dtype=np.int64) * w
    assert offs[-1] > 2**32
    arr = pa.LargeBinaryArray.from_buffers(pa.large_binary(), n, [None, pa.py_buffer(offs), pa.py_buffer(chars.reshape(-1))])
    got = bc.array_sort_indices(_dev(arr, ctx)).to_arrow().to_numpy()
    assert np.array_equal(np.bincount(got.astype(np.int64), minlength=n), np.ones(n, np.int64))  # a permutation
    j = np.sort(rng.choice(n - 1, 1_000_000, replace=False))
    rows = got[j], got[j + 1]
    for a, b, ra, rb in zip(arr.take(pa.array(rows[0])).to_pylist(), arr.take(pa.array(rows[1])).to_pylist(), *rows):
        assert a < b or (a == b and ra < rb)
