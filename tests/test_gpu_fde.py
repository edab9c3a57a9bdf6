"""GPU tests of the first "next" row (SURVEY 8f-1): FDE encoder, FDE candidate scan, candidate-mode MaxSim rerank.

FDE parity is UNPINNED against the reference (its extension's sources are absent, SURVEY F2): the checks here are
(i) bit-exact agreement of the device encoder with the oracle restatement (oracle/fde_oracle.c, same fp32 loop order),
(ii) the scan against numpy, (iii) the rerank against the MaxSim oracle restricted to the same candidates, and
(iv) recall of the true MaxSim top-k among the FDE candidates on planted data."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("CUDA device required", allow_module_level=True)

from morphik_core_b200 import fde  # noqa: E402
from morphik_core_b200.index import MaxSimIndex  # noqa: E402
from oracle import maxsim_oracle as orc  # noqa: E402


def unit_rows(rng, n):
    x = rng.standard_normal((n, 128)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


CFG = fde.FixedDimensionalEncodingConfig()  # the reference's configuration (fast_multivector_store.py:325-331)


def test_config_matches_reference_dimensions():
    assert CFG.fde_dimension == 10240 and CFG.num_partitions == 32
    sh, ai, sg = fde.fde_matrices(CFG)
    assert sh.shape == (20, 128, 5) and ai.shape == (20, 128) and ai.min() >= 0 and ai.max() < 16
    assert set(np.unique(sg).tolist()) == {-1.0, 1.0}
    with pytest.raises(ValueError):
        fde.FixedDimensionalEncodingConfig(final_projection_dimension=100).validate()


def test_encoder_bit_exact_vs_oracle():
    rng = np.random.default_rng(0)
    sh, ai, sg = fde.fde_matrices(CFG)
    idx = MaxSimIndex(dtype="bf16")
    fde.configure_handle(idx, CFG)
    items = [unit_rows(rng, n) for n in (1, 32, 7, 700, 1030, 2500)] + [np.zeros((0, 128), np.float32)]
    for is_doc in (False, True):
        got = fde.encode_items(idx, items, is_doc, CFG.fde_dimension).cpu().numpy()
        for i, x in enumerate(items):
            want = orc.fde_encode_c_proj(x, sh, ai, sg, CFG.scale, is_doc, CFG.projection_dimension)
            assert np.array_equal(got[i], want), (is_doc, i, np.abs(got[i] - want).max())
    # bf16 sources (what the embedding model emits) take the same path
    xb = torch.from_numpy(items[3]).bfloat16()
    got = fde.encode_items(idx, [xb.cuda()], True, CFG.fde_dimension).cpu().numpy()[0]
    want = orc.fde_encode_c_proj(xb.float().numpy(), sh, ai, sg, CFG.scale, True, CFG.projection_dimension)
    assert np.array_equal(got, want)
    # the module-level API of the extension
    q = items[1]
    np.testing.assert_array_equal(fde.generate_query_encoding(q, CFG),
                                  orc.fde_encode_c_proj(q, sh, ai, sg, CFG.scale, False, CFG.projection_dimension))
    np.testing.assert_array_equal(fde.generate_document_encoding(q.tolist(), CFG),
                                  orc.fde_encode_c_proj(q, sh, ai, sg, CFG.scale, True, CFG.projection_dimension))


def test_fde_dot_approximates_chamfer():
    """MUVERA's point: <FDE_q(Q), FDE_doc(P)> tracks the MaxSim (Chamfer) similarity -- rank correlation on random data."""
    rng = np.random.default_rng(1)
    q = unit_rows(rng, 32)
    pages = [unit_rows(rng, 64) for _ in range(200)]
    for j in range(0, 200, 10):  # make some pages related to the query
        pages[j][:32] = q + 0.05 * (j + 1) * rng.standard_normal((32, 128)).astype(np.float32) / 11.3
    qf = fde.generate_query_encoding(q, CFG)
    df = np.stack([fde.generate_document_encoding(p, CFG) for p in pages])
    approx = df @ qf
    exact = orc.float_maxsim_c(q, np.concatenate(pages), orc.page_offsets([64] * 200))
    rel = set(np.argsort(-exact)[:10].tolist())
    assert len(rel & set(np.argsort(-approx)[:30].tolist())) >= 8


@pytest.mark.parametrize("dtype", ["bf16", "int8", "binary"])
def test_two_stage_search_matches_oracle_on_candidates(dtype):
    rng = np.random.default_rng(5)
    lens = [int(x) for x in rng.integers(20, 200, size=300)]
    pages = [unit_rows(rng, n) for n in lens]
    queries = [unit_rows(rng, 32), unit_rows(rng, 20)]
    for qi, q in enumerate(queries):  # plant 6 relevant pages per query
        for j in range(6):
            p = 17 * (qi + 1) + 31 * j
            n = min(len(q), lens[p])
            pages[p][:n] = q[:n] + (0.02 * (j + 1)) * rng.standard_normal((n, 128)).astype(np.float32)
            pages[p] /= np.linalg.norm(pages[p], axis=1, keepdims=True)
    ts_idx = fde.TwoStageIndex(dtype=dtype)
    ts_idx.add_pages(pages[:150])
    ts_idx.add_pages(pages[150:])
    k, n_cand = 5, 40
    cand, cand_scores, cand_counts = ts_idx.candidates(queries, n_cand)
    torch.cuda.synchronize()
    cand = cand.cpu().numpy()
    # (ii) first stage against numpy: cosine scan of the bf16 FDE matrix
    sh, ai, sg = fde.fde_matrices(CFG)
    F = np.stack([orc.bf16_round_np(orc.fde_encode_c_proj(p, sh, ai, sg, CFG.scale, True, 16)) for p in pages])
    inv = 1.0 / np.maximum(np.linalg.norm(F, axis=1), 1e-30)
    for qi, q in enumerate(queries):
        qf = orc.fde_encode_c_proj(q, sh, ai, sg, CFG.scale, False, 16)
        s = (F @ qf) * inv
        want = np.argsort(-s, kind="stable")[:n_cand]
        assert len(set(want.tolist()) & set(cand[qi].tolist())) >= n_cand - 1  # fp32 summation order may swap a near-tie
        np.testing.assert_allclose(cand_scores[qi].cpu().numpy(), np.sort(s)[::-1][:n_cand], rtol=2e-4, atol=1e-5)
    # (iii) rerank == MaxSim oracle restricted to the same candidates (ties -> earlier candidate slot)
    got_s, got_i, got_c = ts_idx.search(queries, k, n_candidates=n_cand)
    rows = np.concatenate(pages)
    off = orc.page_offsets(lens)
    for qi, q in enumerate(queries):
        if dtype == "bf16":
            full = orc.float_maxsim_c(orc.bf16_round_np(q), orc.bf16_round_np(rows), off).astype(np.float64)
        elif dtype == "int8":
            full = orc.int8_maxsim_c(orc.quantize_int8_np(q, 127.0), orc.quantize_int8_np(rows, 127.0), off) / (127.0 * 127.0)
        else:
            full = orc.binary_maxsim_c(orc.sign_pack_c(q), orc.sign_pack_c(rows), off)[0]
        cs = full[cand[qi]]
        order = np.lexsort((np.arange(n_cand), -cs))[:k]
        assert got_i[qi].tolist() == cand[qi][order].tolist(), (dtype, qi)
        np.testing.assert_allclose(got_s[qi], cs[order], rtol=3e-5)
        # (iv) the planted pages are found through the two stages
        planted = {17 * (qi + 1) + 31 * j for j in range(6)}
        assert len(planted & set(got_i[qi].tolist())) >= 4
    # stage names of the reference's own timing log (fast_multivector_store.py:523,534,550,574)
    assert {"encode_query_ms", "ns_query_ms", "load_multivectors_ms", "rerank_scoring_ms"} <= set(ts_idx.last_timing_ms)


def test_rerank_handles_unused_slots_and_empty_pages():
    rng = np.random.default_rng(9)
    pages = [unit_rows(rng, n) for n in (40, 0, 64, 33, 5)]
    ts_idx = fde.TwoStageIndex(dtype="bf16")
    ts_idx.add_pages(pages)
    q = unit_rows(rng, 32)
    cand = torch.tensor([3, -1, 1, 0, -1, 4], dtype=torch.int64, device="cuda")
    ts, ti, tc = ts_idx.rerank(q, cand, k=6)
    torch.cuda.synchronize()
    full = orc.float_maxsim_c(orc.bf16_round_np(q), orc.bf16_round_np(np.concatenate(pages)), orc.page_offsets([40, 0, 64, 33, 5]))
    valid = [3, 1, 0, 4]
    order = sorted(range(4), key=lambda j: (-full[valid[j]], j))
    assert int(tc[0]) == 4 and ti[0][:4].cpu().tolist() == [valid[j] for j in order] and ti[0][4:].cpu().tolist() == [-1, -1]
    np.testing.assert_allclose(ts[0][:4].cpu().numpy(), [full[valid[j]] for j in order], rtol=3e-5, atol=1e-6)


def test_upstream_knobs_fill_empty_partitions_and_final_projection():
    """fill_empty_partitions and final_projection_dimension (upstream config fields the reference leaves at their defaults):
    device encoder bit-exact against the oracle restatement; matrices may also come from a caller (FdeMatrices)."""
    rng = np.random.default_rng(12)
    items = [unit_rows(rng, n) for n in (1, 3, 9, 40, 700, 2500)] + [np.zeros((0, 128), np.float32)]
    for cfg in (fde.FixedDimensionalEncodingConfig(fill_empty_partitions=True),
                fde.FixedDimensionalEncodingConfig(final_projection_dimension=1024),
                fde.FixedDimensionalEncodingConfig(fill_empty_partitions=True, final_projection_dimension=512, num_repetitions=7)):
        m = fde.fde_matrices_full(cfg)
        idx = MaxSimIndex(dtype="bf16")
        fde.configure_handle(idx, cfg, m)
        for is_doc in (False, True):
            got = fde.encode_items(idx, items, is_doc, cfg.fde_dimension).cpu().numpy()
            assert got.shape == (len(items), cfg.fde_dimension)
            for i, x in enumerate(items):
                want = orc.fde_encode_c_ex(x, m.simhash, m.ams_index, m.ams_sign, cfg.scale, is_doc, cfg.projection_dimension,
                                           cfg.fill_empty_partitions, m.final_index, m.final_sign, cfg.final_projection_dimension)
                assert np.array_equal(got[i], want), (cfg, is_doc, i, np.abs(got[i] - want).max())
    # fill_empty: a 3-point document has no all-zero partition block any more
    cfg = fde.FixedDimensionalEncodingConfig(fill_empty_partitions=True)
    m = fde.fde_matrices_full(cfg)
    d = orc.fde_encode_c_ex(items[1], m.simhash, m.ams_index, m.ams_sign, cfg.scale, True, 16, True).reshape(20, 32, 16)
    assert (np.abs(d).sum(axis=2) > 0).all()
    q = orc.fde_encode_c_ex(items[1], m.simhash, m.ams_index, m.ams_sign, cfg.scale, False, 16, True).reshape(20, 32, 16)
    assert ((np.abs(q).sum(axis=2) > 0).sum(axis=1) <= 3).all()  # queries are never filled


@pytest.mark.parametrize("n_q", [1, 3, 16, 17, 32, 50, 80, 100, 130])
def test_fde_scan_tensor_path_matches_simt_and_numpy(n_q):
    """fde_scan_umma_kernel (pages = M, bf16 hi/lo queries = N, the matrix read once per 128 queries) against the SIMT scan
    and numpy: partial last tile, every accumulator-width class (16 / 32 / .. / 128 columns per half), > 128 queries."""
    rng = np.random.default_rng(40 + n_q)
    cfg = fde.FixedDimensionalEncodingConfig()
    n_pages = 128 * 9 + 37
    two = fde.TwoStageIndex(dtype="bf16", config=cfg)
    F = torch.randn((n_pages, cfg.fde_dimension), generator=torch.Generator().manual_seed(n_q)).to(torch.bfloat16)
    F[5] = 0  # an all-zero FDE row (inverse norm 0)
    inv = 1.0 / torch.clamp(F.float().norm(dim=1), min=1e-30)
    inv[5] = 0
    two._grow(n_pages)
    two._F[:n_pages].copy_(F.cuda()); two._inv[:n_pages].copy_(inv.cuda()); two._n = n_pages
    q = torch.randn((n_q, cfg.fde_dimension), generator=torch.Generator().manual_seed(7)).cuda()
    two.index.set_option("fde_gemm", 1)
    a = two.fde_scores(q)[:, :n_pages].cpu().numpy()
    two.index.set_option("fde_gemm", 0)
    b = two.fde_scores(q)[:, :n_pages].cpu().numpy()
    want = (q.cpu().double() @ F.double().T * inv.double()).numpy()
    scale = np.abs(want).max()
    assert np.abs(b - want).max() / scale < 2e-6
    assert np.abs(a - want).max() / scale < 2e-5  # bf16 hi + lo of the query: ~2^-17 relative per term
    assert np.all(a[:, 5] == 0)


def test_two_stage_batched_search_equals_per_query_rerank_and_rebuild():
    rng = np.random.default_rng(55)
    lens = [int(x) for x in rng.integers(32, 200, size=400)]
    pages = [orc.bf16_round_np(unit_rows(rng, n)) for n in lens]  # bf16-valued, like real ColPali embeddings
    queries = [unit_rows(rng, t) for t in (32, 20, 32, 40, 7)]
    two = fde.TwoStageIndex(dtype="bf16")
    two.add_pages(pages)
    s, i, c = two.search(queries, 6, n_candidates=50)
    cand, _, _ = two.candidates(queries, 50)
    torch.cuda.synchronize()
    for qi, q in enumerate(queries):
        ts, ti, tc = two.rerank(q, cand[qi].contiguous(), 6)
        assert i[qi].tolist() == ti[0].cpu().tolist() and np.allclose(s[qi], ts[0].cpu().numpy(), rtol=1e-6)
    # FDE matrix rebuilt from the packed rows (shard-file load path) equals the one built at ingest from the float pages
    F0, inv0 = [t.clone() for t in two.fde_rows()]
    two.rebuild_from_index()
    F1, inv1 = two.fde_rows()
    assert torch.equal(F0.view(torch.int16), F1.view(torch.int16)) and torch.equal(inv0, inv1)
