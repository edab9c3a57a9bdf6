"""Generate the golden fixtures under tests/golden/ by EXECUTING reference code in the build container.

Run from the repo root:  python tests/golden/make_golden.py REFERENCE_CHECKOUT
Needs a checkout of the reference project and transformers; the tests have neither, which is why the outputs
(small .npz / .json files) are committed next to this script.

What is executed:
  * REFERENCE_CHECKOUT/core/utils/fast_ops.py (loaded by file path; HAS_RUST is False here so the authoritative
    pure-Python fallbacks run): binary_quantize, binary_quantize_packed, hamming_distance(_batch).
  * transformers.models.colpali.processing_colpali.ColPaliProcessor.score_retrieval -- the port of
    colpali_engine v0.3.13 ``score_multi_vector`` that the reference calls at
    core/vector_store/fast_multivector_store.py:553-555 (colpali_engine itself is not installed; SURVEY F6).
  * core/vector_store/dual_multivector_store.py (DualMultiVectorStore) over two recording member stores: every call it
    makes on its members and every member attribute it reads (dual_store_calls.json).
The SQL ``max_sim`` (multi_vector_store.py:287-311) cannot be executed (no Postgres): its fixture holds only the
known answers implied by core/tests/unit/test_multivector.py and is marked ``derived``.
"""
import asyncio
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

REF = None  # the reference checkout, from the command line
OUT = os.path.dirname(os.path.abspath(__file__))


def load_fast_ops():
    spec = importlib.util.spec_from_file_location("ref_fast_ops", os.path.join(REF, "core/utils/fast_ops.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.HAS_RUST is False
    return mod


def gen_sign_pack(fo):
    rng = np.random.default_rng(20260922)
    x = rng.standard_normal((96, 128)).astype(np.float32)
    # edge values the Rust tests name (binary_ops.rs:299-306): 0.0 -> 0, plus -0.0, NaN, inf, denormals
    x[0, :8] = [1.0, -0.5, 0.1, -2.0, 0.0, 3.0, -1.0, 0.5]
    x[1, :8] = [1.0, -1.0, 1.0, -1.0, -1.0, 1.0, -1.0, 1.0]  # binary_ops.rs:309-319 -> 0b10100101
    x[2, :6] = [0.0, -0.0, np.nan, np.inf, -np.inf, 1e-45]
    x[3] = 0.0
    packed = np.frombuffer(b"".join(fo.binary_quantize_packed(x)), dtype=np.uint8).reshape(96, 16)
    bools = np.array(fo.binary_quantize(x), dtype=bool)
    # float64 / odd dims go through the same entry point (multi_vector_store.py:334-345)
    x3 = np.array([[0.1, -0.2, 0.3], [-0.1, 0.2, -0.3]])  # test_multivector.py:94-109 -> "101", "010"
    bools3 = np.array(fo.binary_quantize(x3), dtype=bool)
    packed3 = np.frombuffer(b"".join(fo.binary_quantize_packed(x3)), dtype=np.uint8).reshape(2, 1)
    a = rng.integers(0, 256, size=(64, 16), dtype=np.uint8)
    b = rng.integers(0, 256, size=(64, 16), dtype=np.uint8)
    ham = np.array([fo.hamming_distance(bytes(a[i]), bytes(b[i])) for i in range(64)], dtype=np.int64)
    ham_batch = np.array(fo.hamming_distance_batch(bytes(a[0]), [bytes(r) for r in b]), dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "sign_pack.npz"), x=x, packed=packed, bools=bools, x3=x3, bools3=bools3,
                        packed3=packed3, ham_a=a, ham_b=b, ham=ham, ham_batch=ham_batch)


def unit_rows(rng, n, d=128):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def float_maxsim_inputs():
    """The seeded inputs of cases A-E.  float_maxsim.npz stores only what the port computed from them and their digest:
    tests/conftest.py regenerates the inputs with this function and checks the digest before any test uses them."""
    rng = np.random.default_rng(4321)

    def bf16(x):
        return torch.from_numpy(x).bfloat16().float().numpy()

    # case A: equal-length pages (the shape family of every BASELINE config), two queries of different length
    qa = [unit_rows(rng, 32), unit_rows(rng, 20)]
    pa = [unit_rows(rng, 64) for _ in range(12)]
    # case B (and C): ragged pages inside one 128-batch -> zero-padding quirk (max includes the zero rows)
    lens_b = [5, 64, 1, 33, 64, 17, 40, 2]
    pb = [unit_rows(rng, n) for n in lens_b]
    qb = [-np.abs(unit_rows(rng, 8)), unit_rows(rng, 32)]  # first query is all-negative: makes the quirk visible
    pb[0] = np.abs(pb[0])
    pb[2] = np.abs(pb[2])
    # case D: bf16-valued inputs (what the embedding model really emits: colpali_embedding_model.py:262)
    qd = bf16(unit_rows(rng, 32))
    pd = [bf16(unit_rows(rng, 96)) for _ in range(16)]
    # case E: bf16-valued, all-positive pages and a candidate list in first-stage order
    lens_e = [int(x) for x in rng.integers(3, 90, size=40)]
    pe = [bf16(np.abs(unit_rows(rng, n))) for n in lens_e]
    cand_e = rng.permutation(40)[:25]
    qe = [bf16(-np.abs(unit_rows(rng, 20))), bf16(unit_rows(rng, 32))]
    return dict(a_q0=qa[0], a_q1=qa[1], a_pages=np.stack(pa), b_q0=qb[0], b_q1=qb[1], b_rows=np.concatenate(pb),
                b_lens=np.array(lens_b), d_q=qd, d_pages=np.stack(pd), e_rows=np.concatenate(pe), e_lens=np.array(lens_e),
                e_cand=cand_e.astype(np.int64), e_q0=qe[0], e_q1=qe[1])


def inputs_digest(inputs):
    """sha256 over the names, dtypes, shapes and bytes of the inputs."""
    h = hashlib.sha256()
    for name in sorted(inputs):
        a = np.ascontiguousarray(inputs[name])
        h.update(f"{name}:{a.dtype.str}:{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def gen_float_maxsim():
    from transformers.models.colpali.processing_colpali import ColPaliProcessor

    x = float_maxsim_inputs()

    def port(qs, ps, batch_size=128):
        return ColPaliProcessor.score_retrieval(None, [torch.from_numpy(q) for q in qs], [torch.from_numpy(p) for p in ps],
                                                batch_size=batch_size, output_dtype=torch.float32).numpy()

    off_b = np.concatenate([[0], np.cumsum(x["b_lens"])])
    pb = [x["b_rows"][off_b[i]:off_b[i + 1]] for i in range(len(x["b_lens"]))]
    off_e = np.concatenate([[0], np.cumsum(x["e_lens"])])
    pe = [x["e_rows"][off_e[i]:off_e[i + 1]] for i in range(len(x["e_lens"]))]
    out = dict(
        a_scores=port([x["a_q0"], x["a_q1"]], list(x["a_pages"])),
        b_scores=port([x["b_q0"], x["b_q1"]], pb),
        # case C: batch_size smaller than the page count -> padding is per batch, not global
        c_scores=port([x["b_q0"], x["b_q1"]], pb, batch_size=3), c_batch=np.array(3),
        d_scores=port([x["d_q"]], list(x["d_pages"])),
        # case E: the rerank call of FastMultiVectorStore.query_similar (fast_multivector_store.py:553-555): ONE query against
        # the candidate pages in FIRST-STAGE ORDER, one 128-batch (<= 75 candidates) -> the padding quirk follows the list
        e_scores=np.stack([port([q], [pe[int(c)] for c in x["e_cand"]])[0] for q in (x["e_q0"], x["e_q1"])]),
        inputs_sha256=np.array(inputs_digest(x)))
    np.savez_compressed(os.path.join(OUT, "float_maxsim.npz"), **out)


def gen_binary_known_answers():
    """Derived (not executed) known answers for SQL max_sim -- see module docstring."""
    # test_multivector.py:222-256: page1 = 3x[+1]*64,[-1]*64 ; page2 = complement ; query = one row like page1
    e1 = np.ones((3, 128), dtype=np.float32)
    e1[:, 64:] = -1
    e2 = -e1
    q = e1[:1].copy()
    np.savez_compressed(os.path.join(OUT, "binary_known.npz"), pattern_rows=np.concatenate([e1, e2]),
                        pattern_lens=np.array([3, 3]), pattern_query=q, pattern_scores=np.array([1.0, 0.0]),
                        derived=np.array(True))


def gen_dual_store_calls():
    """Run the reference's DualMultiVectorStore, unmodified, over two members that record each call (method, positional and
    keyword arguments) and each attribute read.  Its sibling imports -- the Postgres and Turbopuffer stores, which need
    psycopg / turbopuffer -- are replaced by empty placeholder classes (they are only type annotations there).  The scenario
    is the one tests/test_store_host_logic.py replays: 8 chunks of 4 documents, one query, a lookup, a delete."""
    for pkg in ("core", "core.vector_store", "core.models"):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(REF, *pkg.split("."))]
        sys.modules[pkg] = m

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    load("core.models.chunk", "core/models/chunk.py")
    load("core.vector_store.base_vector_store", "core/vector_store/base_vector_store.py")
    for name, cls in (("fast_multivector_store", "FastMultiVectorStore"), ("multi_vector_store", "MultiVectorStore")):
        stub = types.ModuleType(f"core.vector_store.{name}")
        setattr(stub, cls, type(cls, (), {}))
        sys.modules[f"core.vector_store.{name}"] = stub
    dual_mod = load("core.vector_store.dual_multivector_store", "core/vector_store/dual_multivector_store.py")
    chunk_cls = sys.modules["core.models.chunk"].DocumentChunk

    rng = np.random.default_rng(8)
    chunks = [chunk_cls(document_id=f"d{i // 2}", content=f"c{i}", embedding=rng.standard_normal((3, 128)).astype(np.float32),
                        chunk_number=i % 2, metadata={"i": i}) for i in range(8)]
    query = chunks[5].embedding
    calls = []

    def encode(a):
        if a is chunks:
            return {"ref": "chunks"}
        if a is query:
            return {"ref": "query"}
        if isinstance(a, (list, tuple)):
            return [encode(x) for x in a]
        assert a is None or isinstance(a, (bool, int, str)), type(a)
        return a

    results = {"initialize": True, "store_embeddings": (True, [], {"rows": 0}), "query_similar": [], "get_chunks_by_id": [],
               "delete_chunks_by_document_id": True, "close": None}

    class Member:
        def __init__(self, name):
            self._name = name

        def __getattr__(self, attr):
            if attr not in results:
                calls.append({"member": self._name, "attribute": attr})
                return f"{self._name}.{attr}"

            def call(*args, **kwargs):
                calls.append({"member": self._name, "method": attr, "args": encode(args), "kwargs": {k: encode(v) for k, v in kwargs.items()}})
                if attr in ("initialize", "close"):
                    return results[attr]

                async def done():
                    return results[attr]
                return done()
            return call

    dual = dual_mod.DualMultiVectorStore(fast_store=Member("fast"), slow_store=Member("slow"))
    ops = []

    def step(label, fn):
        del calls[:]
        out = fn()
        if asyncio.iscoroutine(out):
            asyncio.run(out)
        ops.append({"label": label, "calls": list(calls)})

    step("initialize", dual.initialize)
    step("uri", lambda: dual.uri)
    step("storage", lambda: dual.storage)
    step("store_embeddings", lambda: dual.store_embeddings(chunks, app_id="app"))
    step("query_similar", lambda: dual.query_similar(query, 3, None, "app"))
    step("get_chunks_by_id", lambda: dual.get_chunks_by_id([("d1", 0), ("zz", 0)], "app"))
    step("delete_chunks_by_document_id", lambda: dual.delete_chunks_by_document_id("d2", "app"))
    step("query_similar_after_delete", lambda: dual.query_similar(query, 8, None, "app"))
    step("close", dual.close)
    with open(os.path.join(OUT, "dual_store_calls.json"), "w") as f:
        json.dump({"source": "core/vector_store/dual_multivector_store.py", "operations": ops}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    REF = sys.argv[1]
    fo = load_fast_ops()
    gen_sign_pack(fo)
    gen_float_maxsim()
    gen_binary_known_answers()
    gen_dual_store_calls()
    for f in sorted(os.listdir(OUT)):
        if f.endswith((".npz", ".json")):
            print(f, os.path.getsize(os.path.join(OUT, f)))
