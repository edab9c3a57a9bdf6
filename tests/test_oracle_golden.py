"""Pins the oracle (oracle/) against everything the reference offers for this path (SURVEY.md 8c):

* outputs of the reference's own core/utils/fast_ops.py executed in the build container (sign_pack.npz),
* the Rust unit-test vectors morphik_rust/src/binary_ops.rs:299-333,
* core/tests/unit/test_multivector.py:94-109 ("101"/"010"), :166-177 (self-match == T), :222-256 (pattern order),
* outputs of the transformers port of colpali_engine's score_multi_vector (float_maxsim.npz).
"""
import os

import numpy as np
import pytest

from oracle import maxsim_oracle as orc


@pytest.fixture(scope="module")
def sp(golden_dir):
    return np.load(os.path.join(golden_dir, "sign_pack.npz"))


@pytest.fixture(scope="module")
def fm(float_maxsim):
    return float_maxsim


def test_sign_pack_matches_reference_fast_ops(sp):
    for fn in (orc.sign_pack_np, orc.sign_pack_c):
        assert np.array_equal(fn(sp["x"]), sp["packed"])
    # unpacked bool form (fast_ops.binary_quantize) agrees with the packed one
    assert np.array_equal(np.unpackbits(sp["packed"], axis=1, bitorder="big").astype(bool), sp["bools"])


def test_sign_pack_rust_known_answers():
    # binary_ops.rs:299-306: v > 0.0 rule, 0.0 -> false
    v = np.array([[1.0, -0.5, 0.1, -2.0, 0.0, 3.0, -1.0, 0.5]], dtype=np.float32)
    assert orc.sign_pack_c(v)[0, 0] == 0b10100101
    # binary_ops.rs:309-319: [1,-1,1,-1,-1,1,-1,1] -> 0b10100101 (MSB first)
    v = np.array([[1.0, -1.0, 1.0, -1.0, -1.0, 1.0, -1.0, 1.0]], dtype=np.float32)
    assert orc.sign_pack_np(v)[0, 0] == 0b10100101 and orc.sign_pack_c(v)[0, 0] == 0b10100101
    # binary_ops.rs:322-333
    a = np.array([0b11110000, 0b10101010], dtype=np.uint8)
    b = np.array([0b11110000, 0b01010101], dtype=np.uint8)
    assert int(orc.hamming_np(a, b)) == 8
    assert orc.c_oracle().oracle_hamming(a.ctypes.data, b.ctypes.data, 2) == 8


def test_sign_pack_odd_dim_known_answers(sp):
    # test_multivector.py:94-109: [[0.1,-0.2,0.3],[-0.1,0.2,-0.3]] -> "101", "010"; dims not multiple of 8 pad with 0 bits
    got = orc.sign_pack_c(sp["x3"])
    assert np.array_equal(got, sp["packed3"])
    assert np.array_equal(np.unpackbits(got, axis=1, bitorder="big")[:, :3].astype(bool), sp["bools3"])
    assert np.array_equal(sp["bools3"], np.array([[1, 0, 1], [0, 1, 0]], dtype=bool))


def test_special_values(sp):
    # 0.0, -0.0, NaN, -inf -> 0 ; +inf, denormal -> 1
    bits = np.unpackbits(orc.sign_pack_c(sp["x"][2:3]), axis=1, bitorder="big")[0, :6]
    assert bits.tolist() == [0, 0, 0, 1, 0, 1]


def test_hamming_matches_reference(sp):
    assert np.array_equal(orc.hamming_np(sp["ham_a"], sp["ham_b"]), sp["ham"])
    assert np.array_equal(orc.hamming_np(sp["ham_a"][0][None, :], sp["ham_b"]), sp["ham_batch"])
    lib = orc.c_oracle()
    for i in range(len(sp["ham"])):
        a, b = np.ascontiguousarray(sp["ham_a"][i]), np.ascontiguousarray(sp["ham_b"][i])
        assert lib.oracle_hamming(a.ctypes.data, b.ctypes.data, 16) == sp["ham"][i]


def test_binary_maxsim_pattern_known_answer(golden_dir):
    kn = np.load(os.path.join(golden_dir, "binary_known.npz"))
    d = orc.sign_pack_c(kn["pattern_rows"])
    q = orc.sign_pack_c(kn["pattern_query"])
    off = orc.page_offsets(kn["pattern_lens"])
    for fn in (orc.binary_maxsim_np, orc.binary_maxsim_c):
        scores, sim_int = fn(q, d, off)
        assert scores.tolist() == kn["pattern_scores"].tolist() == [1.0, 0.0]
        assert sim_int.tolist() == [128, 0]
    # ORDER BY similarity DESC: pattern page first (test_multivector.py:253-256)
    assert orc.topk_np(scores, 2)[1].tolist() == [0, 1]


def test_binary_maxsim_self_match_is_maximum():
    # test_multivector.py:166-177: a stored page queried with its own vectors ranks first; score == T exactly
    rng = np.random.default_rng(0)
    pages = [rng.uniform(-1, 1, size=(3, 128)).astype(np.float32) for _ in range(6)]
    d = orc.sign_pack_c(np.concatenate(pages))
    off = orc.page_offsets([3] * 6)
    for j in range(6):
        scores, _ = orc.binary_maxsim_c(orc.sign_pack_c(pages[j]), d, off)
        assert scores[j] == 3.0 and scores.max() == 3.0
        ts, ti = orc.topk_c(scores, 6)
        assert ti[0] == j or scores[ti[0]] == 3.0
        assert np.all(np.diff(ts) <= 0)  # non-increasing (test_multivector.py:176-177)


def test_binary_maxsim_c_equals_numpy_and_empty_pages():
    rng = np.random.default_rng(1)
    lens = [0, 7, 1, 0, 33, 64, 5]
    d = rng.integers(0, 256, size=(sum(lens), 16), dtype=np.uint8)
    q = rng.integers(0, 256, size=(11, 16), dtype=np.uint8)
    q[3] = q[2]  # duplicate query vectors count separately (row_number(), multi_vector_store.py:294-296)
    off = orc.page_offsets(lens)
    s_np, i_np = orc.binary_maxsim_np(q, d, off)
    s_c, i_c = orc.binary_maxsim_c(q, d, off)
    assert np.array_equal(s_np, s_c) and np.array_equal(i_np, i_c)
    assert s_c[0] == 0.0 and s_c[3] == 0.0  # COALESCE(..., 0.0)
    assert np.array_equal(s_c, i_c / 128.0)  # score == sim_int / 128 exactly


def test_float_maxsim_equal_length_matches_port(fm):
    rows = fm["a_pages"].reshape(-1, 128)
    off = orc.page_offsets([fm["a_pages"].shape[1]] * fm["a_pages"].shape[0])
    for qi, q in enumerate((fm["a_q0"], fm["a_q1"])):
        for fn in (orc.float_maxsim_np, orc.float_maxsim_c):
            for compat in (False, True):  # equal lengths: both modes coincide
                got = fn(q, rows, off, zero_pad_compat=compat)
                np.testing.assert_allclose(got, fm["a_scores"][qi], rtol=2e-6, atol=2e-6)


def test_float_maxsim_zero_pad_quirk_matches_port(fm):
    off = orc.page_offsets(fm["b_lens"])
    for qi, q in enumerate((fm["b_q0"], fm["b_q1"])):
        for fn in (orc.float_maxsim_np, orc.float_maxsim_c):
            got = fn(q, fm["b_rows"], off, zero_pad_compat=True, batch=128)
            np.testing.assert_allclose(got, fm["b_scores"][qi], rtol=2e-6, atol=2e-6)
            got3 = fn(q, fm["b_rows"], off, zero_pad_compat=True, batch=int(fm["c_batch"]))
            np.testing.assert_allclose(got3, fm["c_scores"][qi], rtol=2e-6, atol=2e-6)
    # the quirk is real: the all-negative query scores 0 on short pages in compat mode, < 0 in clean mode
    clean = orc.float_maxsim_c(fm["b_q0"], fm["b_rows"], off, zero_pad_compat=False)
    compat = orc.float_maxsim_c(fm["b_q0"], fm["b_rows"], off, zero_pad_compat=True)
    assert compat[0] == 0.0 and clean[0] < 0.0
    longest = int(np.argmax(fm["b_lens"]))
    assert clean[longest] == compat[longest]


def test_float_maxsim_rerank_in_candidate_order_matches_port(fm):
    """Case E: the reference's rerank call -- one query against its <= 75 candidates in first-stage order, one batch
    (fast_multivector_store.py:553-555).  The oracle restricted to the candidate pages IN THAT ORDER reproduces the port."""
    off = orc.page_offsets(fm["e_lens"])
    cand = fm["e_cand"]
    sub_rows = np.concatenate([fm["e_rows"][off[c]:off[c + 1]] for c in cand])
    sub_off = orc.page_offsets([int(fm["e_lens"][c]) for c in cand])
    for qi, q in enumerate((fm["e_q0"], fm["e_q1"])):
        got = orc.float_maxsim_c(q, sub_rows, sub_off, zero_pad_compat=True, batch=128)
        np.testing.assert_allclose(got, fm["e_scores"][qi], rtol=2e-6, atol=2e-6)
    longest = max(int(fm["e_lens"][c]) for c in cand)
    assert all((s == 0.0) == (int(fm["e_lens"][c]) < longest) for s, c in zip(fm["e_scores"][0], cand))


def test_float_maxsim_bf16_valued_inputs(fm):
    rows = fm["d_pages"].reshape(-1, 128)
    off = orc.page_offsets([fm["d_pages"].shape[1]] * fm["d_pages"].shape[0])
    got = orc.float_maxsim_c(fm["d_q"], rows, off)
    np.testing.assert_allclose(got, fm["d_scores"][0], rtol=2e-6, atol=2e-6)
    assert np.array_equal(orc.bf16_round_np(rows), rows)  # fixture really is bf16-valued


def test_score_multi_vector_port_is_the_port(fm):
    # the torch restatement used as the bench's reference arm reproduces the fixture bit-for-bit
    lens = fm["b_lens"]
    off = orc.page_offsets(lens)
    ps = [fm["b_rows"][off[i]:off[i + 1]] for i in range(len(lens))]
    got = orc.score_multi_vector_port([fm["b_q0"], fm["b_q1"]], ps, batch_size=128).numpy()
    np.testing.assert_allclose(got, fm["b_scores"], rtol=1e-6, atol=1e-6)
    dense = orc.score_multi_vector_port_dense(fm["a_q0"][None], fm["a_pages"]).numpy()
    np.testing.assert_allclose(dense[0], fm["a_scores"][0], rtol=1e-6, atol=1e-6)


def test_int8_maxsim_c_equals_numpy():
    rng = np.random.default_rng(2)
    lens = [3, 0, 40, 32, 1]
    rows = rng.integers(-127, 128, size=(sum(lens), 128), dtype=np.int8)
    q = rng.integers(-127, 128, size=(9, 128), dtype=np.int8)
    off = orc.page_offsets(lens)
    assert np.array_equal(orc.int8_maxsim_np(q, rows, off), orc.int8_maxsim_c(q, rows, off))


def test_topk_tie_break_and_mask():
    s = np.array([1.0, 3.0, 3.0, 2.0, 3.0, -1.0])
    ts, ti = orc.topk_np(s, 3)
    assert ti.tolist() == [1, 2, 4]
    allow = np.array([1, 0, 1, 1, 1, 1], dtype=bool)
    bits = np.packbits(allow, bitorder="little").view(np.uint8)
    words = np.zeros(1, dtype=np.uint32)
    words[0] = int.from_bytes(bits.tobytes().ljust(4, b"\0"), "little")
    ts_c, ti_c = orc.topk_c(s, 4, words)
    ts_n, ti_n = orc.topk_np(s, 4, allow)
    assert ti_c.tolist() == ti_n.tolist() == [2, 4, 3, 0]
    assert orc.topk_c(s, 10)[1].tolist() == [1, 2, 4, 3, 0, 5]  # fewer than k available
