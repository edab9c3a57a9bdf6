"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI (ctypes), against the oracle.

Bars (SURVEY 8d "Parity gates"): sign bits / Hamming / int8 bit-exact; bf16 scores within 1e-3 relative of the fp32
oracle evaluated on the same bf16-rounded inputs (measured: ~1e-6); top-k id lists identical to the oracle's
(score DESC, page id ASC) on inputs without near-ties, and identical as score multisets otherwise.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover - the gpu marker normally deselects these on CPU boxes
    pytest.skip("CUDA device required", allow_module_level=True)

from morphik_core_b200 import _native as nat  # noqa: E402
from morphik_core_b200.index import MaxSimIndex  # noqa: E402
from oracle import maxsim_oracle as orc  # noqa: E402

BF16_RTOL = 1e-3  # north-star tolerance for bf16 storage


def unit_rows(rng, n, d=128):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def make_pages(rng, lens):
    return [unit_rows(rng, n) if n > 0 else np.zeros((0, 128), np.float32) for n in lens]


def oracle_float(queries, pages, bf16=True):
    rows = np.concatenate(pages) if sum(len(p) for p in pages) else np.zeros((0, 128), np.float32)
    off = orc.page_offsets([len(p) for p in pages])
    rr = orc.bf16_round_np(rows) if bf16 else rows
    return np.stack([orc.float_maxsim_c(orc.bf16_round_np(q) if bf16 else q, rr, off) for q in queries])


def assert_close_rel(got, want, rtol):
    scale = np.maximum(np.abs(want), 1e-3)
    err = np.abs(got - want) / scale
    assert err.max() <= rtol, f"max rel err {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"


# ------------------------------------------------------------------------------------------------ quantiser (a-2)
def test_sign_pack_matches_reference_golden(golden_dir):
    sp = np.load(os.path.join(golden_dir, "sign_pack.npz"))
    idx = MaxSimIndex(dtype="binary")
    got = idx.sign_pack(sp["x"]).cpu().numpy()
    assert np.array_equal(got, sp["packed"])  # bytes produced by the reference's own fast_ops.py
    got_bf16 = idx.sign_pack(torch.from_numpy(sp["x"]).bfloat16().cuda()).cpu().numpy()
    want_bf16 = orc.sign_pack_c(torch.from_numpy(sp["x"]).bfloat16().float().numpy())
    assert np.array_equal(got_bf16, want_bf16)
    big = np.random.default_rng(5).standard_normal((10007, 128)).astype(np.float32)
    assert np.array_equal(idx.sign_pack(big).cpu().numpy(), orc.sign_pack_c(big))


def test_hamming_distance_batch_matches_reference_golden(golden_dir):
    sp = np.load(os.path.join(golden_dir, "sign_pack.npz"))  # ham_batch was produced by the reference's fast_ops.py
    idx = MaxSimIndex(dtype="binary")
    got = idx.hamming_distance_batch(bytes(sp["ham_a"][0]), [bytes(r) for r in sp["ham_b"]]).cpu().numpy()
    assert np.array_equal(got, sp["ham_batch"])
    a = np.array([0b11110000, 0b10101010] + [0] * 14, dtype=np.uint8)  # binary_ops.rs:322-333 -> 8
    b = np.array([[0b11110000, 0b01010101] + [0] * 14], dtype=np.uint8)
    assert idx.hamming_distance_batch(a, b).cpu().tolist() == [8]
    big = np.random.default_rng(0).integers(0, 256, size=(100003, 16), dtype=np.uint8)
    assert np.array_equal(idx.hamming_distance_batch(big[7], big).cpu().numpy(), orc.hamming_np(big[7][None, :], big))
    with pytest.raises(ValueError, match="length mismatch"):
        idx.hamming_distance_batch(b"\x00" * 16, [b"\x00" * 15])


# ------------------------------------------------------------------------------------------------ float MaxSim (a-7)
@pytest.mark.parametrize("dtype", ["bf16", "int8", "fp8"])
def test_host_transports_agree(dtype):
    """b200ms_search_host moves small calls through mapped pinned memory (zero-copy) and batches through the copy engines:
    same kernels, identical results; option zero_copy=0 forces the copy-engine transport."""
    rng = np.random.default_rng(77)
    lens = [1, 31, 32, 33, 0, 64, 127, 128, 129, 700, 1030, 2] + list(rng.integers(1, 400, size=40))
    pages = make_pages(rng, lens)
    a = MaxSimIndex(dtype=dtype); a.add_pages(pages)
    b = MaxSimIndex(dtype=dtype); b.set_option("zero_copy", 0); b.add_pages(pages)
    allowed = rng.random(len(pages)) < 0.5
    for qs in ([unit_rows(rng, 32)], [unit_rows(rng, 5)], [unit_rows(rng, t) for t in (32, 7, 40, 1)],
               [unit_rows(rng, 32) for _ in range(12)]):  # 12 x 32 = 384 rows: above the zero-copy threshold on both
        for mask in (None, a.mask_from_pages(allowed)):
            ra, rb = a.search_host(qs, k=9, allow_mask=mask), b.search_host(qs, k=9, allow_mask=mask)
            assert all(np.array_equal(x, y) for x, y in zip(ra, rb))


def test_bf16_config0_shape_single_query():
    # BASELINE config 0: 100 pages x 1024 patches x 128-d, one 32-token query
    rng = np.random.default_rng(1234)
    pages = make_pages(rng, [1024] * 100)
    q = [unit_rows(np.random.default_rng(4321), 32)]
    idx = MaxSimIndex(dtype="bf16")
    idx.add_pages(pages)
    got = idx.score_matrix(q)
    want = oracle_float(q, pages)
    assert_close_rel(got, want, 2e-5)  # same bf16-rounded inputs, fp32 accumulate: only summation order differs
    want_fp32 = oracle_float(q, pages, bf16=False)  # vs the reference's fp32 inputs: bf16 storage error only
    assert_close_rel(got, want_fp32, BF16_RTOL)
    ts, ti, tc = idx.search_host(q, k=10)
    os_, oi = orc.topk_np(want[0], 10)
    assert tc[0] == 10 and ti[0].tolist() == oi.tolist()
    np.testing.assert_allclose(ts[0], os_, rtol=2e-5)


def test_bf16_golden_fixture_from_score_multi_vector(float_maxsim):
    fm = float_maxsim
    # case D is bf16-valued (what ColQwen emits), so bf16 storage is lossless and the port's scores are the target
    idx = MaxSimIndex(dtype="bf16")
    idx.add_pages(list(fm["d_pages"]))
    got = idx.score_matrix([fm["d_q"]])
    np.testing.assert_allclose(got[0], fm["d_scores"][0], rtol=2e-5, atol=1e-5)
    # case A (fp32-valued, equal lengths): within the bf16 tolerance of the port's fp32 result
    idx2 = MaxSimIndex(dtype="bf16")
    idx2.add_pages(list(fm["a_pages"]))
    got2 = idx2.score_matrix([fm["a_q0"], fm["a_q1"]])
    assert_close_rel(got2, fm["a_scores"], BF16_RTOL)


@pytest.mark.parametrize("unit_rows_", [0, 64, 1000])
def test_bf16_ragged_pages_empty_pages_unit_boundaries(unit_rows_):
    rng = np.random.default_rng(7)
    lens = [1, 31, 32, 33, 0, 64, 127, 128, 129, 5, 700, 1030, 0, 2, 96, 255, 256, 257, 40, 1] + list(
        rng.integers(1, 300, size=60))
    pages = make_pages(rng, lens)
    queries = [unit_rows(rng, 32), unit_rows(rng, 7), -np.abs(unit_rows(rng, 20))]  # last: all-negative dots possible
    idx = MaxSimIndex(dtype="bf16")
    if unit_rows_:
        idx.set_tuning(unit_rows=unit_rows_)
    idx.add_pages(pages[:30])
    idx.add_pages(pages[30:])  # incremental append
    got = idx.score_matrix(queries)
    want = oracle_float(queries, pages)
    assert_close_rel(got, want, 2e-5)
    assert np.all(got[:, [4, 12]] == 0.0)  # empty pages score exactly 0


@pytest.mark.parametrize("dtype", ["bf16", "int8"])
def test_one_cta_forms_match_oracle(dtype):
    """pair_cta = 0 (what a partition without whole TPCs falls back to): NM = 1 / 2 two-warpgroup kernel and the NM = 4 / 8
    four-warpgroup kernel against the oracle -- bf16 within rounding, int8 bit-exact."""
    rng = np.random.default_rng(808)
    lens = [1, 33, 0, 64, 700, 1030, 2] + list(rng.integers(1, 300, size=50))
    pages = make_pages(rng, lens)
    rows = np.concatenate(pages)
    off = orc.page_offsets(lens)
    for n_q in (1, 5, 13, 32, 40):  # 1, 2, 4, 8 (int8: NM=8), 10 query tiles
        queries = [unit_rows(rng, 32 if i % 2 else 29) for i in range(n_q)]
        a = MaxSimIndex(dtype=dtype); a.set_option("pair_cta", 0); a.set_option("unit_rows", 400); a.add_pages(pages)
        got = a.score_matrix(queries)
        if dtype == "bf16":
            assert_close_rel(got, oracle_float(queries, pages), 3e-5)
        else:
            rq = orc.quantize_int8_np(rows, 127.0)
            want = np.stack([orc.int8_maxsim_c(orc.quantize_int8_np(q, 127.0), rq, off) for q in queries])
            assert np.array_equal(np.rint(got * 127.0 * 127.0).astype(np.int64), want), n_q


@pytest.mark.parametrize("dtype", ["bf16", "int8", "fp8"])
@pytest.mark.parametrize("unit_rows_,n_pages", [(400, 57), (64, 9), (4096, 3), (400, 1)])
def test_cta_pair_form_agrees(dtype, unit_rows_, n_pages):
    """The CTA-pair kernel (tcgen05 cta_group::2, two unit streams per pair) is bit-identical to the one-CTA kernels:
    odd/even unit counts, fewer units than CTAs, a single page, phantom query tiles, int8 with NM = 8."""
    rng = np.random.default_rng(909 + n_pages)
    lens = ([1, 33, 0, 64, 700, 1030, 2] + list(rng.integers(1, 300, size=50)))[:n_pages]
    pages = make_pages(rng, lens)
    for n_q in (5, 9, 13, 32, 40, 70):  # 2 (pair_cta = 2 only), 3, 4, 8, 10, 18 query tiles
        queries = [unit_rows(rng, 32 if i % 2 else 29) for i in range(n_q)]
        a = MaxSimIndex(dtype=dtype); a.set_option("pair_cta", 2); a.set_option("unit_rows", unit_rows_); a.add_pages(pages)
        b = MaxSimIndex(dtype=dtype); b.set_option("pair_cta", 0); b.set_option("unit_rows", unit_rows_); b.add_pages(pages)
        ga, gb = a.score_matrix(queries), b.score_matrix(queries)
        assert np.array_equal(ga, gb), (dtype, n_q, np.abs(ga - gb).max())
        if dtype == "bf16" and n_q == 13:
            assert_close_rel(ga, oracle_float(queries, pages), 3e-5)


@pytest.mark.parametrize("dtype", ["bf16", "int8", "fp8", "binary"])
@pytest.mark.parametrize("unit_rows_,n_pages", [(400, 70), (64, 9), (4096, 70), (400, 1), (0, 400)])
def test_rows_as_m_kernel_is_bit_identical_to_query_as_m(dtype, unit_rows_, n_pages):
    """maxsim_rowm_kernel (lone query: patch rows = M operand, four epilogue warps, cross-warp page combine in shared memory)
    against the query-as-M kernels it replaces for scans of <= 2 query groups: 1 and 2 groups, short last groups, pages of
    1 .. 1030 rows (pages inside one chunk, pages crossing tiles and units), empty pages, one page only, more units than SMs."""
    rng = np.random.default_rng(1234 + n_pages)
    base = [1, 31, 32, 33, 0, 64, 127, 128, 129, 5, 700, 1030, 0, 2, 96, 255, 256, 257, 40, 1]
    lens = (base + list(rng.integers(1, 300, size=400)))[:n_pages] if n_pages > 1 else [333]
    if n_pages == 400:
        lens = list(rng.integers(1, 1100, size=400))
    pages = make_pages(rng, lens)
    a = MaxSimIndex(dtype=dtype); a.set_option("rowm", 1)
    b = MaxSimIndex(dtype=dtype); b.set_option("rowm", 0)
    if dtype == "binary":
        b.set_option("b1_tensor", 0)  # the POPC kernel: an independent formulation
    for ix in (a, b):
        if unit_rows_:
            ix.set_option("unit_rows", unit_rows_)
        ix.add_pages(pages)
    for qs in ([unit_rows(rng, 32)], [unit_rows(rng, 7)], [-np.abs(unit_rows(rng, 20))], [unit_rows(rng, 64)],
               [unit_rows(rng, 45)], [unit_rows(rng, 32), unit_rows(rng, 3)]):
        ga, gb = a.score_matrix(qs), b.score_matrix(qs)
        assert np.array_equal(ga, gb), (dtype, [len(q) for q in qs], np.abs(ga - gb).max(), np.argwhere(ga != gb)[:5])
        ta, tb = a.search_host(qs, k=7), b.search_host(qs, k=7)
        assert np.array_equal(ta[1], tb[1]) and np.array_equal(ta[0], tb[0])
    if dtype == "bf16":
        qs = [unit_rows(rng, 32), unit_rows(rng, 30)]
        assert_close_rel(a.score_matrix(qs), oracle_float(qs, pages), 3e-5)
        for ix in (a, b):
            ix.set_option("zero_pad_compat", 16)
        q1 = [-np.abs(unit_rows(rng, 20))]
        assert np.array_equal(a.score_matrix(q1), b.score_matrix(q1))


@pytest.mark.parametrize("dtype", ["bf16", "binary"])
def test_rows_as_m_kernel_flushes_finished_pages_early(dtype):
    """One CTA, 64-row work units: a 128-row page gives lane quadrants 2 and 3 a partial maximum, then 400 pages of <= 64 rows
    follow whose tiles only fill quadrants 0 and 1 -- those warps must hand the finished page over at the next block, not at
    their next chunk (which never comes), or the 128-slot page table wraps around under them."""
    rng = np.random.default_rng(99)
    lens = [128] + [int(x) for x in rng.integers(33, 65, size=400)] + [128] + [40] * 300
    pages = make_pages(rng, lens)
    a = MaxSimIndex(dtype=dtype); a.set_option("rowm", 1)
    b = MaxSimIndex(dtype=dtype); b.set_option("rowm", 0)
    if dtype == "binary":
        b.set_option("b1_tensor", 0)
    for ix in (a, b):
        ix.set_tuning(unit_rows=64, max_ctas=1)
        ix.add_pages(pages)
    for qs in ([unit_rows(rng, 32)], [unit_rows(rng, 9)]):
        ga, gb = a.score_matrix(qs), b.score_matrix(qs)
        assert np.array_equal(ga, gb), (dtype, np.argwhere(ga != gb)[:5])


def test_rows_as_m_kernel_binary_matches_oracle_on_uniform_pages():
    """1024-row pages (the BASELINE shape): every page spans 8 tiles and all four epilogue warps; exact integers."""
    rng = np.random.default_rng(77)
    lens = [1024] * 300
    pages = make_pages(rng, lens)
    idx = MaxSimIndex(dtype="binary"); idx.add_pages(pages)
    q = [unit_rows(rng, 32)]
    got = idx.score_matrix(q)
    want, _ = orc.binary_maxsim_c(orc.sign_pack_c(q[0]), orc.sign_pack_c(np.concatenate(pages)), orc.page_offsets(lens))
    assert np.array_equal(got[0], want)


def test_cta_pair_form_large_and_topk():
    """Pair kernel on a corpus that gives every pair many units (persistent loop, stage ring wrap, dummy tail tiles)."""
    rng = np.random.default_rng(4242)
    lens = list(rng.integers(900, 1100, size=700))
    pages = make_pages(rng, lens)
    queries = [unit_rows(rng, 32) for _ in range(32)]
    a = MaxSimIndex(dtype="bf16"); a.set_option("pair_cta", 1); a.add_pages(pages)
    b = MaxSimIndex(dtype="bf16"); b.set_option("pair_cta", 0); b.add_pages(pages)
    assert np.array_equal(a.score_matrix(queries), b.score_matrix(queries))
    ta, tb = a.search_host(queries, k=10), b.search_host(queries, k=10)
    assert np.array_equal(ta[1], tb[1]) and np.array_equal(ta[0], tb[0])


@pytest.mark.parametrize("n_q,t", [(2, 32), (3, 32), (5, 17), (8, 32), (16, 32), (32, 32), (33, 20), (1, 70), (2, 1030)])
def test_bf16_query_batches_and_long_queries(n_q, t):
    rng = np.random.default_rng(100 + n_q * 7 + t)
    lens = list(rng.integers(20, 200, size=40)) + [1024, 1024]
    pages = make_pages(rng, lens)
    queries = [unit_rows(rng, t if i % 2 == 0 else max(1, t - 3)) for i in range(n_q)]
    idx = MaxSimIndex(dtype="bf16")
    idx.set_tuning(unit_rows=512)
    idx.add_pages(pages)
    got = idx.score_matrix(queries)
    want = oracle_float(queries, pages)
    assert_close_rel(got, want, 3e-5)
    k = 7
    ts, ti, tc = idx.search_host(queries, k=k)
    for q in range(n_q):
        _, oi = orc.topk_np(want[q], k)
        assert ti[q].tolist() == oi.tolist(), f"query {q}"


# ------------------------------------------------------------------------------------------------ int8 MaxSim (config 3)
@pytest.mark.parametrize("n_q", [1, 4, 9, 32])
def test_int8_bit_exact(n_q):
    rng = np.random.default_rng(11 + n_q)
    lens = [1, 33, 0, 64, 200, 1024, 17, 96] + list(rng.integers(1, 260, size=30))
    pages = make_pages(rng, lens)
    queries = [unit_rows(rng, 32 if i % 3 else 19) for i in range(n_q)]
    # every dot product of these tokens is negative (all-negative query x all-positive pages below), so every per-chunk maximum
    # is a negative int32: the epilogue's integer max must order those exactly (a float max over the bit patterns would not)
    queries[0] = -np.abs(queries[0])
    for j in (3, 4, 9):
        pages[j] = np.abs(pages[j])
    idx = MaxSimIndex(dtype="int8", i8_scale=127.0)
    idx.set_tuning(unit_rows=256)
    idx.add_pages(pages)
    scores, goff, n_pages, _ = idx.score_groups(queries)
    torch.cuda.synchronize()
    raw = scores[:, :n_pages].cpu().numpy().astype(np.int64)
    rows_q = orc.quantize_int8_np(np.concatenate(pages), 127.0)
    # the packed corpus holds exactly the oracle's quantisation (rint half-even, clamp)
    packed = idx.packed_rows().cpu().numpy().view(np.int8)
    off_pad = np.concatenate([[0], np.cumsum([(n + 31) // 32 * 32 for n in lens])])
    off = orc.page_offsets(lens)
    for p in (0, 1, 5, 7):
        assert np.array_equal(packed[off_pad[p]:off_pad[p] + lens[p]], rows_q[off[p]:off[p + 1]])
    for qi, q in enumerate(queries):
        want = orc.int8_maxsim_c(orc.quantize_int8_np(q, 127.0), rows_q, off)
        got = raw[goff[qi]:goff[qi + 1]].sum(axis=0)
        assert np.array_equal(got, want), f"query {qi}"  # integer arithmetic: bit-exact
        if qi == 0:
            assert want[[3, 4, 9]].max() < 0  # the negative-maximum case really occurred
    ts, ti, tc = idx.search_host(queries, k=5)
    for qi, q in enumerate(queries):
        want = orc.int8_maxsim_c(orc.quantize_int8_np(q, 127.0), rows_q, off)
        _, oi = orc.topk_np(want, 5)
        assert ti[qi].tolist() == oi.tolist()


# ------------------------------------------------------------------------------------------------ binary MaxSim (a-3, a-4)
def test_binary_known_answers_from_reference_tests(golden_dir):
    kn = np.load(os.path.join(golden_dir, "binary_known.npz"))
    idx = MaxSimIndex(dtype="binary")
    idx.add_pages([kn["pattern_rows"][:3], kn["pattern_rows"][3:]])
    ts, ti, tc = idx.search_host([kn["pattern_query"]], k=2)
    assert ti[0].tolist() == [0, 1] and ts[0].tolist() == [1.0, 0.0]  # test_multivector.py:222-256
    rng = np.random.default_rng(3)
    pages = [rng.uniform(-1, 1, size=(3, 128)).astype(np.float32) for _ in range(9)]
    idx2 = MaxSimIndex(dtype="binary")
    idx2.add_pages(pages)
    for j in (0, 4, 8):  # self-match is top-1 with score exactly T (test_multivector.py:166-177)
        ts, ti, tc = idx2.search_host([pages[j]], k=9)
        assert ti[0][0] == j and ts[0][0] == 3.0 and np.all(np.diff(ts[0]) <= 0)


# 0 = POPC kernel, 1 = tcgen05 kernels, 2 = auto.  With the default rowm = 1, paths 1 and 2 send a scan of ONE 32-token group
# to the rows-as-M kernel (maxsim_rowm.cu); "query_as_m" is path 1 with rowm = 0, so that scan runs on maxsim_b1_umma_kernel<1>.
@pytest.mark.parametrize("path", [0, 1, 2, "query_as_m"])
@pytest.mark.parametrize("n_q", [1, 3, 8, 13])
def test_binary_bit_exact(n_q, path):
    rng = np.random.default_rng(50 + n_q)
    lens = [1, 31, 32, 33, 0, 64, 1024, 5, 700] + list(rng.integers(1, 200, size=50))
    pages = make_pages(rng, lens)
    queries = [unit_rows(rng, t) for t in ([32, 7, 45, 1, 20, 64, 33, 32, 2, 9, 100, 31, 32][:n_q])]
    idx = MaxSimIndex(dtype="binary")
    if path == "query_as_m":
        idx.set_option("rowm", 0)
        path = 1
    idx.set_option("b1_tensor", path)
    idx.add_pages(pages)
    got = idx.score_matrix(queries)
    d_bits = orc.sign_pack_c(np.concatenate(pages))
    off = orc.page_offsets(lens)
    for qi, q in enumerate(queries):
        want, want_int = orc.binary_maxsim_c(orc.sign_pack_c(q), d_bits, off)
        assert np.array_equal(got[qi], want), f"query {qi}"  # multiples of 1/128: exact
    ts, ti, tc = idx.search_host(queries, k=6)
    for qi, q in enumerate(queries):
        want, _ = orc.binary_maxsim_c(orc.sign_pack_c(q), d_bits, off)
        os_, oi = orc.topk_np(want, 6)
        assert ti[qi].tolist() == oi.tolist() and np.array_equal(ts[qi].astype(np.float64), os_)


# ------------------------------------------------------------------------------------------------ top-k / filter
def test_topk_ties_mask_and_short_lists():
    rng = np.random.default_rng(9)
    # binary scores are multiples of 1/128 -> many exact ties: the tie rule (lower page id first) must hold
    pages = [np.sign(rng.standard_normal((4, 128))).astype(np.float32) for _ in range(300)]
    pages += [pages[3].copy(), pages[3].copy()]  # exact duplicates of page 3 at ids 300, 301
    q = [pages[3][:2]]
    idx = MaxSimIndex(dtype="binary")
    idx.add_pages(pages)
    d_bits = orc.sign_pack_c(np.concatenate(pages))
    off = orc.page_offsets([4] * len(pages))
    want, _ = orc.binary_maxsim_c(orc.sign_pack_c(q[0]), d_bits, off)
    for k in (1, 3, 50, 302, 400):
        ts, ti, tc = idx.search_host(q, k=k)
        os_, oi = orc.topk_np(want, k)
        n = min(k, len(pages))
        assert tc[0] == n and ti[0][:n].tolist() == oi.tolist()
        assert np.all(ti[0][n:] == -1) and np.all(np.isinf(ts[0][n:]))
    assert ti[0][:3].tolist() == [3, 300, 301]
    allowed = rng.random(len(pages)) < 0.3
    allowed[3] = False
    allowed[300] = True
    ts, ti, tc = idx.search_host(q, k=20, allow_mask=idx.mask_from_pages(allowed))
    os_, oi = orc.topk_np(want, 20, allowed)
    assert ti[0].tolist() == oi.tolist() and ti[0][0] == 300
    none = np.zeros(len(pages), dtype=bool)
    ts, ti, tc = idx.search_host(q, k=5, allow_mask=idx.mask_from_pages(none))
    assert tc[0] == 0 and np.all(ti[0] == -1)


def test_topk_large_k_and_many_pages_bf16():
    rng = np.random.default_rng(21)
    pages = make_pages(rng, [32] * 5000)
    queries = [unit_rows(rng, 32) for _ in range(3)]
    idx = MaxSimIndex(dtype="bf16")
    idx.add_pages(pages)
    got = idx.score_matrix(queries)
    for k in (1000, 4096):
        ts, ti, tc = idx.search_host(queries, k=k)
        for q in range(3):
            # compare against a ranking of the GPU's own scores (isolates the selection from fp rounding)
            os_, oi = orc.topk_np(got[q].astype(np.float32), k)
            assert ti[q].tolist() == oi.tolist()
            np.testing.assert_array_equal(ts[q], os_.astype(np.float32))


def test_merge_topk_matches_oracle():
    rng = np.random.default_rng(33)
    idx = MaxSimIndex(dtype="bf16")
    n_q, m, k = 5, 800, 100
    s = rng.standard_normal((n_q, m)).astype(np.float32)
    s[:, 100:140] = s[:, 0:40]  # ties across "shards"
    ids = np.stack([rng.permutation(100000)[:m] for _ in range(n_q)]).astype(np.int64)
    ids[:, -17:] = -1  # unused slots
    ts, ti, tc = idx.merge_topk(torch.from_numpy(s).cuda(), torch.from_numpy(ids).cuda(), k)
    ts, ti = ts.cpu().numpy(), ti.cpu().numpy()
    for q in range(n_q):
        valid = ids[q] >= 0
        order = np.lexsort((ids[q][valid], -s[q][valid].astype(np.float64)))[:k]
        assert ti[q].tolist() == ids[q][valid][order].tolist()
        np.testing.assert_array_equal(ts[q], s[q][valid][order])


# ------------------------------------------------------------------------------------------------ size-independent properties
def test_properties_at_scale_bf16():
    """At a size the oracle cannot sweep in seconds (16k pages x 1024 patches, 4 GiB bf16), check invariants of MaxSim."""
    n_pages, p = 16384, 1024
    g = torch.Generator(device="cuda").manual_seed(1234)
    rows = torch.randn((n_pages * p, 128), generator=g, device="cuda", dtype=torch.float32)
    rows = torch.nn.functional.normalize(rows, dim=1).to(torch.bfloat16)
    qg = torch.Generator(device="cuda").manual_seed(4321)
    q = torch.nn.functional.normalize(torch.randn((32, 128), generator=qg, device="cuda"), dim=1)
    # plant: page 777's first 32 rows are the query tokens themselves -> score ~ 32 (the maximum), rank 1
    rows[777 * p: 777 * p + 32] = q.to(torch.bfloat16)
    # duplicate page 5 into page 9000 -> identical scores; reverse the row order of page 42 into page 43 -> identical
    rows[9000 * p:9001 * p] = rows[5 * p:6 * p]
    rows[43 * p:44 * p] = rows[42 * p:43 * p].flip(0)
    buf = torch.empty(rows.numel() * 2 + 1024, dtype=torch.uint8, device="cuda")
    off = (-buf.data_ptr()) % 1024
    packed = buf[off:off + rows.numel() * 2]
    packed.copy_(rows.view(torch.uint8).reshape(-1))
    idx = MaxSimIndex(dtype="bf16")
    idx.adopt_packed(packed, [p] * n_pages)
    qn = q.cpu().numpy()
    s = idx.score_matrix([qn])[0]
    assert s.argmax() == 777 and abs(s[777] - 32.0) < 0.05
    assert s[9000] == s[5] and s[43] == s[42]
    # oracle on a bounded sample of pages (every 512th + the special ones)
    sample = sorted(set(range(0, n_pages, 512)) | {5, 42, 43, 777, 9000})
    rows_h = torch.stack([rows[i * p:(i + 1) * p].float().cpu() for i in sample]).numpy().reshape(-1, 128)
    want = orc.float_maxsim_c(orc.bf16_round_np(qn), rows_h, orc.page_offsets([p] * len(sample)))
    assert_close_rel(s[sample], want, 2e-5)
    # linearity in the query scale: scoring 2q doubles every score exactly (power-of-two scaling is exact in bf16/fp32)
    s2 = idx.score_matrix([2.0 * qn])[0]
    assert np.array_equal(s2, 2.0 * s)
    # batch consistency: the same query inside a 32-query batch (NM=4, two passes) gives the same scores
    others = [torch.nn.functional.normalize(torch.randn((32, 128), generator=qg, device="cuda"), dim=1).cpu().numpy() for _ in range(31)]
    sb = idx.score_matrix([qn] + others)
    assert np.array_equal(sb[0], s)
    ts, ti, tc = idx.search_host([qn] + others, k=10)
    assert ti[0][0] == 777
    for qi in range(32):
        _, oi = orc.topk_np(sb[qi].astype(np.float32), 10)
        assert ti[qi].tolist() == oi.tolist()


@pytest.mark.parametrize("dtype", ["binary", "int8"])
def test_sliced_topk_is_exact_with_ties_and_large_ints(dtype):
    """Corpora above 16384 pages use the two-level top-k (per-slice select + raw-key merge): the result must equal the
    oracle's global (score DESC, id ASC) order -- including exact ties (binary) and int scores above 2^24 (int8)."""
    rng = np.random.default_rng(123)
    n_pages = 40000
    base = np.sign(rng.standard_normal((n_pages * 32, 128))).astype(np.float32)
    base[base == 0] = 1.0
    if dtype == "int8":
        base *= rng.uniform(0.5, 1.0, size=(n_pages * 32, 1)).astype(np.float32)
    # many duplicate pages -> exact ties spread over different slices
    base[32 * 30000:32 * 30100] = base[32 * 100:32 * 200]
    base[32 * 39900:32 * 40000] = base[32 * 100:32 * 200]
    rows = torch.from_numpy(base).cuda()
    idx = MaxSimIndex(dtype=dtype)
    step = 5000
    for p0 in range(0, n_pages, step):
        idx.add_pages(list(rows[p0 * 32:(p0 + step) * 32].view(step, 32, 128)))
    queries = [base[32 * 150:32 * 150 + 32].copy(), np.sign(rng.standard_normal((20, 128))).astype(np.float32)]
    got = idx.score_matrix(queries)
    for k in (10, 1000, 4096):
        ts, ti, tc = idx.search_host(queries, k=k)
        for qi in range(2):
            os_, oi = orc.topk_np(got[qi], k)  # scores are exact integers / multiples of 1/128: ranking them is the oracle order
            assert ti[qi].tolist() == oi.tolist(), (dtype, k, qi)
    off = orc.page_offsets([32] * n_pages)
    if dtype == "binary":
        want, _ = orc.binary_maxsim_c(orc.sign_pack_c(queries[0]), orc.sign_pack_c(base), off)
        assert np.array_equal(got[0], want)
    else:
        want = orc.int8_maxsim_c(orc.quantize_int8_np(queries[0], 127.0), orc.quantize_int8_np(base, 127.0), off)
        assert np.array_equal(np.rint(got[0] * 127.0 * 127.0).astype(np.int64), want) and want.max() > (1 << 24)


@pytest.mark.parametrize("dtype", ["int8", "binary"])
def test_properties_at_scale_int8_binary(dtype):
    """16384 pages x 1024 patches (int8 2 GiB / 1-bit 256 MiB): invariants + oracle on a sample, single query and a batch
    (the batch takes the tensor-core 1-bit path and the sliced top-k)."""
    n_pages, p = 16384, 1024
    g = torch.Generator(device="cuda").manual_seed(99)
    rows = torch.nn.functional.normalize(torch.randn((n_pages * p, 128), generator=g, device="cuda"), dim=1)
    q = torch.nn.functional.normalize(torch.randn((32, 128), generator=g, device="cuda"), dim=1)
    rows[4242 * p: 4242 * p + 32] = q  # planted: contains the query tokens verbatim -> maximum score, rank 1
    rows[9000 * p:9001 * p] = rows[5 * p:6 * p]  # duplicate page -> identical score
    rows[43 * p:44 * p] = rows[42 * p:43 * p].flip(0)  # permuted rows -> identical score
    idx = MaxSimIndex(dtype=dtype)
    step = 2048
    for p0 in range(0, n_pages, step):
        idx.add_pages(list(rows[p0 * p:(p0 + step) * p].view(step, p, 128)))
    qn = q.cpu().numpy()
    others = [torch.nn.functional.normalize(torch.randn((32, 128), generator=g, device="cuda"), dim=1).cpu().numpy() for _ in range(7)]
    s1 = idx.score_matrix([qn])[0]
    sb = idx.score_matrix([qn] + others)
    assert np.array_equal(sb[0], s1)  # same query alone (POPC / NM=1) and inside a batch (tensor path / NM=2): bit-identical
    assert s1.argmax() == 4242 and s1[9000] == s1[5] and s1[43] == s1[42]
    if dtype == "binary":
        assert s1[4242] == 32.0  # every token finds itself: Hamming 0
    sample = sorted(set(range(0, n_pages, 1024)) | {5, 42, 43, 4242, 9000})
    rows_h = torch.stack([rows[i * p:(i + 1) * p].cpu() for i in sample]).numpy().reshape(-1, 128)
    off = orc.page_offsets([p] * len(sample))
    if dtype == "binary":
        want = orc.binary_maxsim_c(orc.sign_pack_c(qn), orc.sign_pack_c(rows_h), off)[0]
        assert np.array_equal(s1[sample], want)
    else:
        want = orc.int8_maxsim_c(orc.quantize_int8_np(qn, 127.0), orc.quantize_int8_np(rows_h, 127.0), off)
        assert np.array_equal(np.rint(s1[sample] * 127.0 * 127.0).astype(np.int64), want)
    ts, ti, tc = idx.search_host([qn] + others, k=10)
    for qi in range(8):
        _, oi = orc.topk_np(sb[qi], 10)
        assert ti[qi].tolist() == oi.tolist()
    assert ti[0][0] == 4242


# ------------------------------------------------------------------------------------------------ fp8 e4m3 corpora (config-2 sweep point)
def oracle_fp8(queries, pages, scale=64.0):
    rows = np.concatenate(pages) if sum(len(p) for p in pages) else np.zeros((0, 128), np.float32)
    off = orc.page_offsets([len(p) for p in pages])
    rr = orc.dequantize_e4m3_np(orc.quantize_e4m3_np(rows, scale))
    return np.stack([orc.float_maxsim_c(orc.dequantize_e4m3_np(orc.quantize_e4m3_np(q, scale)), rr, off) for q in queries]) / (scale * scale)


@pytest.mark.parametrize("n_q", [1, 5, 13, 40])
def test_fp8_matches_oracle(n_q):
    """B200MS_F8: e4m3(x * 64) rows and queries, tcgen05 kind::f8f6f4 with fp32 accumulation.  The packed bytes equal the
    oracle's round-to-nearest-even e4m3 codes; scores match the oracle's fp32 MaxSim of the dequantised values."""
    rng = np.random.default_rng(300 + n_q)
    lens = [1, 33, 0, 64, 200, 1024, 17, 96] + list(rng.integers(1, 260, size=30))
    pages = make_pages(rng, lens)
    pages[2 + 1][0, :4] = [7.5, -9.0, 1e-4, 0.0]  # saturation (7.5*64 > 448), subnormals, zero
    queries = [unit_rows(rng, 32 if i % 3 else 19) for i in range(n_q)]
    idx = MaxSimIndex(dtype="fp8")
    assert idx.i8_scale == 64.0 and idx.row_bytes == 128
    idx.set_tuning(unit_rows=256)
    idx.add_pages(pages)
    packed = idx.packed_rows().cpu().numpy()
    codes = orc.quantize_e4m3_np(np.concatenate(pages), 64.0)
    off_pad = np.concatenate([[0], np.cumsum([(n + 31) // 32 * 32 for n in lens])])
    off = orc.page_offsets(lens)
    for p in (0, 1, 3, 5, 7):
        assert np.array_equal(packed[off_pad[p]:off_pad[p] + lens[p]], codes[off[p]:off[p + 1]])
    got = idx.score_matrix(queries)
    want = oracle_fp8(queries, pages)
    assert_close_rel(got, want, 1e-4)  # products of e4m3 values are exact in fp32; only the summation order differs
    ts, ti, tc = idx.search_host(queries, k=5)
    for qi in range(n_q):
        assert ti[qi].tolist() == orc.topk_np(got[qi].astype(np.float32), 5)[1].tolist()
    # vs the unquantised fp32 MaxSim: the quantisation error of e4m3 (3 mantissa bits) stays within a few percent
    full = oracle_float(queries, pages, bf16=False)
    live = np.abs(full) > 0.5
    live[:, 3] = False  # page 3 carries the deliberately saturated / subnormal row
    assert (np.abs(got - full)[live] / np.abs(full)[live]).max() < 0.08


# ------------------------------------------------------------------------------------------------ zero_pad_compat (SURVEY App. A.2)
@pytest.mark.parametrize("case,batch", [("b", 128), ("c", 3)])
def test_zero_pad_compat_matches_score_multi_vector_golden(float_maxsim, case, batch):
    """Product option zero_pad_compat=<batch size> reproduces colpali_engine score_multi_vector's padding quirk (a page
    shorter than the longest of its batch scores max(true, 0) per token): golden cases B (one 128-batch) and C
    (batch_size=3) were produced by the transformers port of score_multi_vector (tests/golden/make_golden.py)."""
    fm = float_maxsim
    lens = fm["b_lens"].tolist()
    off = orc.page_offsets(lens)
    pages = [fm["b_rows"][off[i]:off[i + 1]] for i in range(len(lens))]
    queries = [fm["b_q0"], fm["b_q1"]]
    want = fm[f"{case}_scores"]
    idx = MaxSimIndex(dtype="bf16")
    idx.set_option("zero_pad_compat", batch)
    idx.add_pages(pages)
    got = idx.score_matrix(queries)
    assert_close_rel(got, want, BF16_RTOL)
    # the quirk is visible: the all-negative query's clean MaxSim differs on the short pages
    clean = MaxSimIndex(dtype="bf16"); clean.add_pages(pages)
    assert np.abs(clean.score_matrix(queries)[0] - want[0]).max() > 0.1
    # and against the oracle's own switch on bf16-rounded inputs (tight tolerance), batches of queries too (pair kernel)
    many = queries + [unit_rows(np.random.default_rng(5), 32) * (-1 if i % 2 else 1) for i in range(11)]
    rr = orc.bf16_round_np(fm["b_rows"])
    want2 = np.stack([orc.float_maxsim_c(orc.bf16_round_np(q), rr, off, zero_pad_compat=True, batch=batch) for q in many])
    assert_close_rel(idx.score_matrix(many), want2, 3e-5)
    for pc in (0, 2):  # one-CTA and CTA-pair forms agree bit for bit
        alt = MaxSimIndex(dtype="bf16"); alt.set_option("zero_pad_compat", batch); alt.set_option("pair_cta", pc); alt.add_pages(pages)
        assert np.array_equal(alt.score_matrix(many), idx.score_matrix(many))


def test_zero_pad_compat_rerank_batches_candidates_like_the_reference():
    """In the two-stage path the reference scores ONE batch of <= 75 candidates in first-stage order
    (fast_multivector_store.py:529,553-555): the clamp follows the candidate list, not the page ids."""
    rng = np.random.default_rng(61)
    lens = [int(x) for x in rng.integers(3, 90, size=40)]
    pages = [np.abs(unit_rows(rng, n)) for n in lens]
    q = -np.abs(unit_rows(rng, 20))  # every true maximum is negative: clamped pages score exactly 0
    idx = MaxSimIndex(dtype="bf16")
    idx.set_option("zero_pad_compat", 128)
    idx.add_pages(pages)
    cand = [17, 3, 29, 8, 11, 30, 2]
    ci = torch.tensor([cand, cand[::-1]], dtype=torch.int64, device="cuda")
    qd = torch.from_numpy(np.concatenate([q, q])).cuda()
    ts, ti, tc = idx.rerank_batch(qd, [20, 20], ci, k=len(cand))
    torch.cuda.synchronize()
    sub = [pages[c] for c in cand]
    want = orc.float_maxsim_c(orc.bf16_round_np(q), orc.bf16_round_np(np.concatenate(sub)),
                              orc.page_offsets([len(p) for p in sub]), zero_pad_compat=True, batch=128)
    longest = max(lens[c] for c in cand)
    assert all((w == 0.0) == (lens[c] < longest) for w, c in zip(want, cand))
    for row in range(2):
        order = cand if row == 0 else cand[::-1]
        w = {c: want[cand.index(c)] for c in cand}
        exp = sorted(range(len(order)), key=lambda j: (-w[order[j]], j))
        assert ti[row].cpu().tolist() == [order[j] for j in exp]
        np.testing.assert_allclose(ts[row].cpu().numpy(), [w[order[j]] for j in exp], rtol=3e-5, atol=1e-6)


def test_zero_pad_compat_rerank_matches_port_golden(float_maxsim):
    """Golden case E (produced by the transformers port of score_multi_vector): the reference's rerank call, candidates in
    first-stage order -- b200ms_rerank_batch_device with zero_pad_compat=128 returns the port's scores and ranking."""
    fm = float_maxsim
    lens = fm["e_lens"].tolist()
    off = orc.page_offsets(lens)
    pages = [fm["e_rows"][off[i]:off[i + 1]] for i in range(len(lens))]
    cand = fm["e_cand"]
    idx = MaxSimIndex(dtype="bf16")  # inputs are bf16-valued: storage is lossless
    idx.set_option("zero_pad_compat", 128)
    idx.add_pages(pages)
    qs = [fm["e_q0"], fm["e_q1"]]
    ci = torch.from_numpy(np.stack([cand, cand])).cuda()
    ts, ti, tc = idx.rerank_batch(torch.from_numpy(np.concatenate(qs)).cuda(), [len(q) for q in qs], ci, k=len(cand))
    torch.cuda.synchronize()
    for qi in range(2):
        want = fm["e_scores"][qi]
        order = sorted(range(len(cand)), key=lambda j: (-want[j], j))
        assert ti[qi].cpu().tolist() == [int(cand[j]) for j in order]
        np.testing.assert_allclose(ts[qi].cpu().numpy(), want[order], rtol=2e-5, atol=2e-5)


# ------------------------------------------------------------------------------------------------ batched rerank (per-query lists)
@pytest.mark.parametrize("dtype", ["bf16", "int8", "binary"])
def test_rerank_batch_per_query_candidate_lists(dtype):
    rng = np.random.default_rng(71)
    lens = [int(x) for x in rng.integers(1, 200, size=120)] + [0, 1024]
    pages = make_pages(rng, lens)
    t_list = [32, 7, 40, 32, 1, 33, 64, 20, 32]  # queries of 1-2 groups: tiles shared by several queries and straddled
    queries = [unit_rows(rng, t) for t in t_list]
    idx = MaxSimIndex(dtype=dtype)
    idx.add_pages(pages)
    full = idx.score_matrix(queries)
    n_cand, k = 37, 10
    cand = np.stack([rng.permutation(len(pages))[:n_cand] for _ in queries]).astype(np.int64)
    cand[1, 5] = cand[4, 0] = cand[4, 36] = -1  # unused slots
    qd = torch.from_numpy(np.concatenate(queries)).cuda()
    ts, ti, tc = idx.rerank_batch(qd, t_list, torch.from_numpy(cand).cuda(), k)
    torch.cuda.synchronize()
    ts, ti, tc = ts.cpu().numpy(), ti.cpu().numpy(), tc.cpu().numpy()
    for qi in range(len(queries)):
        valid = [j for j in range(n_cand) if cand[qi, j] >= 0]
        order = sorted(valid, key=lambda j: (-full[qi, cand[qi, j]], j))[:k]
        assert tc[qi] == len(order) and ti[qi][:len(order)].tolist() == [int(cand[qi, j]) for j in order], (dtype, qi)
        np.testing.assert_allclose(ts[qi][:len(order)], [full[qi, cand[qi, j]] for j in order], rtol=1e-6)


# ------------------------------------------------------------------------------------------------ pipelined sharded search, world = 1
def test_sharded_search_pipeline_world1_matches_search():
    """b200ms_sharded_search_begin/_end and the *_host_* forms with a one-rank communicator: same answer as
    b200ms_search_device, two tickets in flight, results one step late."""
    rng = np.random.default_rng(81)
    pages = make_pages(rng, list(rng.integers(1, 200, size=300)))
    idx = MaxSimIndex(dtype="bf16")
    idx.add_pages(pages)
    idx.comm_init(b"\0" * 128, 0, 1)
    batches = [[unit_rows(rng, 32) for _ in range(nq)] for nq in (3, 12, 1, 5)]
    base = 7 << 40
    want = [idx.search_host(b, k=8, id_base=base) for b in batches]
    outs, tickets = [], []
    for b in batches:  # at most two in flight: end(i-1) right after begin(i)
        qd = torch.from_numpy(np.concatenate(b)).cuda()
        out = (torch.empty((len(b), 8), device="cuda"), torch.empty((len(b), 8), dtype=torch.int64, device="cuda"),
               torch.empty((len(b),), dtype=torch.int32, device="cuda"))
        tickets.append(idx.sharded_search_begin(qd, [len(x) for x in b], 8, base, out))
        outs.append(out)
        if len(tickets) >= 2:
            idx.sharded_search_end(tickets[-2])
    idx.sharded_search_end(tickets[-1])
    torch.cuda.synchronize()
    for (ws, wi, wc), (ts, ti, tc) in zip(want, outs):
        assert np.array_equal(ti.cpu().numpy(), wi) and np.array_equal(ts.cpu().numpy(), ws) and np.array_equal(tc.cpu().numpy(), wc)
    # host pipeline
    t_prev, prev = None, None
    for b, (ws, wi, wc) in zip(batches, want):
        qh = torch.from_numpy(np.concatenate(b)).pin_memory()
        t = idx.sharded_search_host_begin(qh, [len(x) for x in b], 8, base)
        if t_prev is not None:
            o = (torch.empty((len(prev[0]), 8)), torch.empty((len(prev[0]), 8), dtype=torch.int64), torch.empty((len(prev[0]),), dtype=torch.int32))
            idx.sharded_search_host_end(t_prev, *o)
            assert np.array_equal(o[1].numpy(), prev[1][1]) and np.array_equal(o[0].numpy(), prev[1][0])
        t_prev, prev = t, (b, (ws, wi, wc))
    o = (torch.empty((len(prev[0]), 8)), torch.empty((len(prev[0]), 8), dtype=torch.int64), torch.empty((len(prev[0]),), dtype=torch.int32))
    idx.sharded_search_host_end(t_prev, *o)
    assert np.array_equal(o[1].numpy(), prev[1][1]) and np.array_equal(o[2].numpy(), prev[1][2])


@pytest.mark.parametrize("dtype", ["bf16", "binary"])
def test_host_graph_replay_matches_plain_launches(dtype):
    """Small unmasked host searches of a repeated shape are captured into a CUDA graph on their second call and replayed
    afterwards; results equal the plain launches, and a corpus change / option change invalidates the graph."""
    rng = np.random.default_rng(91)
    pages = make_pages(rng, list(rng.integers(1, 300, size=150)))
    a = MaxSimIndex(dtype=dtype); a.add_pages(pages)
    b = MaxSimIndex(dtype=dtype); b.set_option("host_graph", 0); b.add_pages(pages)
    qs = [[unit_rows(rng, 32)] for _ in range(6)] + [[unit_rows(rng, 20), unit_rows(rng, 32)] for _ in range(4)]
    l0 = a.launch_count()
    for q in qs:  # same shape repeatedly: warm, capture, replay, replay, ...
        ra, rb = a.search_host(q, k=7), b.search_host(q, k=7)
        assert all(np.array_equal(x, y) for x, y in zip(ra, rb))
    assert a.launch_count() - l0 >= 3 * len(qs)  # replays are counted: pack + score + top-k per call
    extra = make_pages(rng, [64, 200, 1])
    a.add_pages(extra); b.add_pages(extra)  # corpus re-attached: the captured graph must not be replayed
    for q in qs[:4]:
        ra, rb = a.search_host(q, k=7), b.search_host(q, k=7)
        assert all(np.array_equal(x, y) for x, y in zip(ra, rb))
    if dtype == "bf16":
        a.set_option("zero_pad_compat", 128); b.set_option("zero_pad_compat", 128)
        for q in qs[:4]:
            ra, rb = a.search_host(q, k=7), b.search_host(q, k=7)
            assert all(np.array_equal(x, y) for x, y in zip(ra, rb))
