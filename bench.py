#!/usr/bin/env python
"""bench.py -- patch-vectors/sec of the ColPali MaxSim hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path (one JSON line on rank 0)
  python bench.py --impl reference [...]                          # the reference's own CPU formulation, same metric
  python bench.py --dump-outputs DIR [...]                        # + the last timed step's top-k as DIR/<name>.npy

Workload (config.workload): a RESIDENT SHARD of BASELINE configs[1] -- "1M pages x 1024 patches x 128-d bf16, batch-32
queries" needs 262 GB, more than one B200's HBM (SURVEY F7) -- i.e. `--pages` pages per GPU (default 524288 = 137.4 GB of
bf16 patch vectors, the largest shard that leaves room for the scratch; ~1090x the 126 MB L2, so no flush is needed between
iterations) scored against a batch of 32 queries x 32 tokens, top-10 per query.  A "step" = one pass of the hot path over the
whole shard for the whole batch: pack queries -> MaxSim scan (tcgen05) -> top-k (-> all-gather + merge at N > 1).
Synthetic, seeded, unit-norm rows with planted relevant pages; the first `--topic-pages` pages of every shard follow a
topic model (graded relevance) so that two-stage recall against the exhaustive ranking means something.

value   whole-job patch-vectors/s with the query batch already resident in HBM, CUDA events, max over ranks.
        N = 1: b200ms_search_device.  N > 1: b200ms_sharded_search_begin/_end -- local scan + top-k written into the exchange
        layout, ONE ncclAllGather + merge on the handle's communication stream, two steps in flight.
e2e     same metric through the C-ABI with HOST buffers, host clock, max over ranks.  N = 1: b200ms_search_host (pinned host
        query buffer -> H2D -> scan -> top-k -> D2H, synchronous per call).  N > 1: b200ms_sharded_search_host_begin/_end
        (every step copies its queries H2D and its merged top-k D2H; results are collected one step later).
roofline  dominant kernel = maxsim_umma_pair; configs[1] has 1024 resident query tokens => tensor-bound (SURVEY 8d);
          achieved = 2*rows*128*1024 flop per step / CUDA-event time of the scoring launches inside the timed region
legs (each with achieved / peak / bound and an oracle check; see DESIGN.md section 5):
  hbm_regime      the same shard, ONE 32-token query (the HBM-bound regime of the north star's 70 % target)
  config2_sweep   bytes-per-score sweep on a sub-shard: bf16 256 B, int8 128 B, fp8 128 B, 1-bit 16 B per patch vector
  config3_bq256   B_q = 256 (8192 query tokens, 8 CTA-pair passes) through the same (sharded) path
  config4_two_stage  FDE candidates + MaxSim rerank top-1000: p50 / p95 latency, recall@{75,1000} vs the exhaustive ranking
  config0_latency configs[0]: 100 pages, one query, per-call latency of b200ms_search_host vs the CPU formulation
  cpu_baseline    colpali_engine's score_multi_vector formulation (oracle/maxsim_oracle.py: torch einsum, all host cores) on
                  the first pages OF THE SAME SHARD; its scores double as the oracle of `topk_match` (all 32 queries)
  multi_gpu_check (N > 1, before timing) identical merged lists on every rank, planted top-1 found, and a sharded search
                  over a gathered sample checked against the oracle
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

P_PATCH, DIM, T_TOK = 1024, 128, 32
METRIC = "patch_vectors_per_sec_maxsim"
UNIT = "patch-vectors/s"
N_TOPICS, N_ANCHORS = 256, 16


def load_traffic():
    """dram__bytes_read+write per patch vector of the dominant kernel, from the committed ncu --set full capture
    (profiles/<round>/traffic.json, written by tools/ncu_summary.py); None if no capture is committed."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    if os.path.isdir(pdir):
        for rnd in sorted(os.listdir(pdir)):
            path = os.path.join(pdir, rnd, "traffic.json")
            if os.path.exists(path):
                with open(path) as f:
                    best = json.load(f)
    return best


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "tflops_burst": float(p["bf16_tflops"]),
                "tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for t, line in self.rows:
            if not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_mhz_min": sm[0] if sm else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ synthetic workload
def make_queries(n_q: int, seed: int = 4321):
    import torch

    g = torch.Generator().manual_seed(seed)
    q = torch.randn((n_q * T_TOK, DIM), generator=g, dtype=torch.float32)
    return torch.nn.functional.normalize(q, dim=1).contiguous()  # host, [n_q*32, 128]


def topic_anchors(device, seed: int = 777):
    """[N_TOPICS, N_ANCHORS, 128] unit anchor vectors shared by every rank (the 'visual vocabulary' of the topic model)."""
    import torch

    g = torch.Generator(device=device).manual_seed(seed)
    a = torch.randn((N_TOPICS, N_ANCHORS, DIM), generator=g, device=device)
    return torch.nn.functional.normalize(a, dim=2)


def make_topic_queries(n_q: int, anchors, seed: int = 99):
    """Queries about a topic: 32 tokens = that topic's anchors (each twice) + noise, unit norm.  Returns (host [n_q*32,128], topics)."""
    import torch

    g = torch.Generator().manual_seed(seed)
    topics = torch.randint(0, N_TOPICS, (n_q,), generator=g)
    a = anchors.cpu()[topics]  # [n_q, 16, 128]
    toks = a.repeat(1, 2, 1) + 0.35 / DIM ** 0.5 * torch.randn((n_q, T_TOK, DIM), generator=g)
    return torch.nn.functional.normalize(toks, dim=2).reshape(n_q * T_TOK, DIM).contiguous(), topics.tolist()


def build_shard(n_pages: int, device, seed: int, q_host, planted_per_query: int = 10, topic_pages: int = 0, anchors=None):
    """[n_pages*1024, 128] bf16 unit-norm rows in a 1024-aligned buffer; a few pages per query get 64 noisy copies of the
    query's tokens so that the top-k is meaningful (SURVEY 8d 'Synthetic inputs').  The first `topic_pages` pages follow a
    topic model instead of pure noise: page p has topic p % N_TOPICS, covers a random ~60 % of the topic's 16 anchors and has a
    noise level that grows with p // N_TOPICS; half of its rows are covered anchors + noise, the rest background -- MaxSim and FDE
    similarity to a topic query both depend on coverage and noise, so 'recall of the exhaustive top-k among the FDE candidates'
    is a graded, non-trivial number."""
    import torch

    rows_total = n_pages * P_PATCH
    buf = torch.empty(rows_total * DIM * 2 + 1024, dtype=torch.uint8, device=device)
    off = (-buf.data_ptr()) % 1024
    packed = buf[off:off + rows_total * DIM * 2]
    rows = packed.view(torch.bfloat16).view(rows_total, DIM)
    g = torch.Generator(device=device).manual_seed(seed)
    chunk_pages = 2048
    for p0 in range(0, n_pages, chunk_pages):
        n = min(chunk_pages, n_pages - p0)
        x = torch.randn((n * P_PATCH, DIM), generator=g, device=device, dtype=torch.float32)
        if p0 < topic_pages and anchors is not None:
            nt = min(n, topic_pages - p0)
            pid = torch.arange(p0, p0 + nt, device=device)
            topic = pid % N_TOPICS
            level = (pid // N_TOPICS).float() / max(1, (topic_pages + N_TOPICS - 1) // N_TOPICS)  # 0 .. <1
            sigma = (0.25 + 1.75 * level) / DIM ** 0.5  # per-page noise: graded relevance inside a topic
            a = anchors[topic]  # [nt, 16, 128]
            # row r of a page: odd rows are background noise (real pages are not all on topic); even rows carry anchor
            # (r // 2) % 16 of the page's topic -- if the page COVERS that anchor (each page covers a random ~60 % of them),
            # so relevance is graded two ways: how many of the query's tokens a page can answer, and how noisily
            r_idx = torch.arange(P_PATCH, device=device)
            anchor_of_row = (r_idx // 2) % N_ANCHORS
            cover = torch.rand((nt, N_ANCHORS), generator=g, device=device) < 0.6
            on_topic = ((r_idx % 2 == 0)[None, :] & cover[:, anchor_of_row]).reshape(nt * P_PATCH)
            base = a[:, anchor_of_row, :].reshape(nt * P_PATCH, DIM)
            xt = x[: nt * P_PATCH]
            xt.mul_(torch.where(on_topic, sigma.repeat_interleave(P_PATCH), torch.ones((), device=device))[:, None])
            xt.add_(base * on_topic[:, None])
        rows[p0 * P_PATCH:(p0 + n) * P_PATCH] = torch.nn.functional.normalize(x, dim=1).to(torch.bfloat16)
        del x
    n_q = q_host.shape[0] // T_TOK
    qd = q_host.to(device)
    planted = {}
    pg = torch.Generator().manual_seed(seed + 99)
    for qi in range(n_q):
        ids = torch.randint(max(topic_pages, 0) if topic_pages < n_pages else 0, n_pages, (planted_per_query,), generator=pg).tolist()
        planted[qi] = ids
        for j, p in enumerate(ids):
            noise = torch.randn((2 * T_TOK, DIM), generator=g, device=device) * (0.3 / DIM ** 0.5) * (1 + j)
            toks = qd[qi * T_TOK:(qi + 1) * T_TOK].repeat(2, 1) + noise
            rows[p * P_PATCH:p * P_PATCH + 2 * T_TOK] = torch.nn.functional.normalize(toks, dim=1).to(torch.bfloat16)
    return packed, planted


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
def set_cpu_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs are meant to use the host's cores (physical cores by default)."""
    import torch

    want = int(os.environ.get("B200MS_CPU_THREADS", "0")) or max(1, (os.cpu_count() or 2) // 2)
    if torch.get_num_threads() != want:
        torch.set_num_threads(want)
    try:  # the C oracle (OpenMP) reads OMP_NUM_THREADS=1 under torchrun too: lift it for the checker legs
        import ctypes

        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(want))
    except Exception:  # noqa: BLE001
        pass


def cpu_reference_rate(n_q: int, budget_s: float, seed: int = 1234, pages_np=None, q_np=None):
    """patch-vectors/s of the reference's float scorer (score_multi_vector: pad + einsum + max + sum, batch 128) on the host
    CPU with all torch threads, on a bounded sample of the workload: `pages_np` ([C,1024,128] fp32, rows of the GPU shard) when
    given, else freshly generated pages of the same family.  Returns the scores too (they are the oracle of topk_match)."""
    import torch

    from oracle import maxsim_oracle as orc

    set_cpu_threads()
    q = make_queries(n_q).view(n_q, T_TOK, DIM).numpy() if q_np is None else q_np
    g = torch.Generator().manual_seed(seed)

    def sample(n_pages):
        x = torch.randn((n_pages, P_PATCH, DIM), generator=g, dtype=torch.float32)
        return torch.nn.functional.normalize(x, dim=2).bfloat16().float().numpy()  # bf16-valued like the GPU shard

    if pages_np is None:
        probe = sample(32)
        t0 = time.perf_counter()
        orc.score_multi_vector_port_dense(q, probe)
        t_probe = time.perf_counter() - t0
        t0 = time.perf_counter()
        orc.score_multi_vector_port_dense(q, probe)
        t_probe = min(t_probe, time.perf_counter() - t0)
        n_pages = int(max(32, min(4096, 32 * budget_s / max(t_probe, 1e-4))))
        n_pages = max(128, n_pages // 128 * 128) if n_pages >= 128 else n_pages
        pages_np = sample(n_pages)
    else:
        orc.score_multi_vector_port_dense(q, pages_np[:128])  # warm the thread pool
    n_pages = pages_np.shape[0]
    t0 = time.perf_counter()
    scores = orc.score_multi_vector_port_dense(q, pages_np)
    dt = time.perf_counter() - t0
    return {"value": n_pages * P_PATCH / dt, "seconds": dt, "pages": n_pages, "threads": torch.get_num_threads(),
            "checksum": float(scores.sum()), "scores": scores.numpy()}


def config0_latency(packed, q_pin, out_pin, k, skip_cpu, n_pages=100, iters=300):
    """BASELINE configs[0] (N=100 pages x 1024 x 128, B_q=1, T=32): per-call latency of b200ms_search_host on the first
    100 pages of the shard (host query in, host top-k out), and the reference's CPU formulation on the same shapes."""
    import numpy as np
    import torch

    from morphik_core_b200.index import MaxSimIndex

    idx0 = MaxSimIndex(device=packed.device.index or 0, dtype="bf16")
    idx0.adopt_packed(packed[: n_pages * P_PATCH * DIM * 2], [P_PATCH] * n_pages)
    q1 = q_pin[:T_TOK]
    o = (out_pin[0][:1], out_pin[1][:1], out_pin[2][:1])
    out = {"workload": f"configs[0]: {n_pages} pages x {P_PATCH} patches x {DIM}-d bf16, 1 query x {T_TOK} tokens, top-{k}",
           "api": "b200ms_search_host (host query in, host top-k out)", "calls": iters}
    for label, zc, gr in (("", 1, 1), ("no_graph_", 1, 0), ("copy_engine_", 0, 0)):
        idx0.set_option("zero_copy", zc)
        idx0.set_option("host_graph", gr)
        for _ in range(20):
            idx0.search_host_flat(q1, [T_TOK], k, *o)
        lat = []
        for _ in range(iters):
            t0 = time.perf_counter()
            idx0.search_host_flat(q1, [T_TOK], k, *o)
            lat.append(time.perf_counter() - t0)
        lat = np.sort(np.asarray(lat)) * 1e6
        out[label + "e2e_p50_us"] = float(lat[len(lat) // 2])
        out[label + "e2e_p95_us"] = float(lat[int(len(lat) * 0.95)])
    kern = idx0.score_times_ms(64)
    out["scoring_kernel_us"] = 1e3 * sum(kern) / len(kern)
    out["transport"] = ("default: query + metadata written to a mapped pinned block the kernels read in place, results written back the same way, "
                        "pack -> score -> top-k replayed as ONE CUDA graph; no_graph_* = the same with three plain launches; "
                        "copy_engine_* = cudaMemcpyAsync H2D / D2H")
    if not skip_cpu:
        from oracle import maxsim_oracle as orc

        set_cpu_threads()
        qn = q1.view(1, T_TOK, DIM).numpy()
        pages = packed[: n_pages * P_PATCH * DIM * 2].view(torch.bfloat16).view(n_pages, P_PATCH, DIM).float().cpu().numpy()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            orc.score_multi_vector_port_dense(qn, pages)
            ts.append(time.perf_counter() - t0)
        out["cpu_reference_formulation_ms"] = 1e3 * sorted(ts)[len(ts) // 2]
        out["cpu_threads"] = torch.get_num_threads()
    idx0.close()
    return out


def topk_match_from_scores(packed, q_pin, n_q, k, cpu_scores, n_pages):
    """'top-k match vs reference' (BASELINE metric): b200ms_search_host over the first n_pages of the shard, all n_q queries,
    against the CPU formulation's scores of exactly those pages (cpu_baseline's own output).  The CPU side scored the
    bf16-valued rows with bf16-rounded queries in fp32, i.e. the same inputs the kernel sees."""
    import numpy as np

    from morphik_core_b200.index import MaxSimIndex
    from oracle import maxsim_oracle as orc

    sub = MaxSimIndex(device=packed.device.index or 0, dtype="bf16")
    sub.adopt_packed(packed[: n_pages * P_PATCH * DIM * 2], [P_PATCH] * n_pages)
    queries = [q_pin[i * T_TOK:(i + 1) * T_TOK].numpy() for i in range(n_q)]
    ts, ti, tc = sub.search_host(queries, k)
    same, err = 0, 0.0
    for i in range(n_q):
        ws, wi = orc.topk_np(cpu_scores[i], k)
        same += int(ti[i].tolist() == wi.tolist())
        err = max(err, float(np.max(np.abs(ts[i] - ws) / np.maximum(np.abs(ws), 1e-6))))
    sub.close()
    return {"sample": f"first {n_pages} pages of the shard x all {n_q} queries, top-{k}; oracle = the cpu_baseline run's scores",
            "id_lists_identical": f"{same}/{n_q}", "max_rel_score_err": err, "tolerance": 1e-3}


def torch_gpu_reference_rate(rows_bf16, q_dev, n_q, sample_pages=4096, iters=5):
    """The kernel-to-beat on the same GPU (SURVEY 8d): the reference's OWN GPU formulation -- colpali_engine
    score_multi_vector with device="cuda" (fast_multivector_store.py:339,553-555) = einsum("bnd,csd->bcns").max(3).sum(2)
    over 128-page batches -- on a resident sample of the shard (no H2D), in bf16 and in fp32 (TF32 allowed, as the reference
    enables it, colpali_embedding_model.py:32-35).  A reported baseline only; nothing here is on the product path."""
    import torch

    out = {}
    pages = rows_bf16[: sample_pages * P_PATCH].view(sample_pages, P_PATCH, DIM)
    q = q_dev.view(n_q, T_TOK, DIM)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        for name, dt in (("bf16", torch.bfloat16), ("fp32_tf32", torch.float32)):
            qq = q.to(dt)

            def once():
                acc = []
                for j in range(0, sample_pages, 128):
                    pb = pages[j:j + 128].to(dt)
                    acc.append(torch.einsum("bnd,csd->bcns", qq, pb).max(dim=3)[0].sum(dim=2))
                return torch.cat(acc, dim=1)

            once()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                scores = once()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out[name] = {"value": sample_pages * P_PATCH / (ms * 1e-3), "unit": UNIT, "ms": ms,
                         "checksum": float(scores.float().sum())}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    out["sample"] = f"{sample_pages} resident pages x {P_PATCH} patches, {n_q} queries x {T_TOK} tokens, torch.einsum+max+sum, batch 128"
    return out


def run_reference(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_q = args.bq
    vals = []
    for _ in range(args.warmup):
        cpu_reference_rate(n_q, budget_s=min(args.ref_budget, 2.0))
    for _ in range(args.steps):
        vals.append(cpu_reference_rate(n_q, budget_s=args.ref_budget))
    total_pv = sum(v["pages"] * P_PATCH for v in vals)
    total_s = sum(v["seconds"] for v in vals)
    value = total_pv / total_s
    sample = f"{vals[-1]['pages']} pages x {P_PATCH} patches x {DIM}-d (bf16-valued fp32) per step, {n_q} queries x {T_TOK} tokens"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, per_gpu_pages=vals[-1]["pages"], note="CPU arm scores a bounded sample per step"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": vals[-1]["threads"], "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, per_gpu_pages, note=None):
    cfg = {
        "workload": f"configs[1] resident shard: {per_gpu_pages} pages/GPU x {P_PATCH} patches x {DIM}-d bf16, "
                    f"batch-{args.bq} queries x {T_TOK} tokens, top-{args.k} (full config = 1M pages = 262 GB > one B200's HBM)",
        "pages_per_gpu": per_gpu_pages, "patches_per_page": P_PATCH, "dim": DIM, "query_batch": args.bq,
        "query_tokens": T_TOK, "k": args.k, "parallelism": f"document-sharded x{args.gpus}",
        "l2": "inputs larger than L2 (shard >> 126 MB), no flush between iterations",
    }
    if note:
        cfg["note"] = note
    return cfg


# ------------------------------------------------------------------------------------------------ sub-shards in other dtypes
def quantised_subshard(packed_bf16, n_pages, dtype, device_index):
    """A MaxSimIndex of `dtype` over the first n_pages pages of the bf16 shard, converted on the GPU by b200ms_pack_pages."""
    import ctypes

    import torch

    from morphik_core_b200 import _native as nat
    from morphik_core_b200.index import MaxSimIndex, _aligned_bytes

    idx = MaxSimIndex(device=device_index, dtype=dtype)
    buf = _aligned_bytes(n_pages * P_PATCH * idx.row_bytes, idx.device)
    step = 16384
    lens_c = nat.i32_array([P_PATCH] * step)
    with torch.cuda.device(idx.device):
        for p0 in range(0, n_pages, step):
            n = min(step, n_pages - p0)
            src = packed_bf16[p0 * P_PATCH * 256:]
            dst = buf[p0 * P_PATCH * idx.row_bytes:]
            idx.h.check(nat.lib.b200ms_pack_pages(idx.h.ptr, ctypes.c_void_p(src.data_ptr()), nat.BF16, lens_c, n,
                                                  ctypes.c_void_p(dst.data_ptr()), idx.dtype, ctypes.c_float(idx.i8_scale),
                                                  idx._stream()), "b200ms_pack_pages")
    torch.cuda.synchronize(idx.device)
    idx.adopt_packed(buf, [P_PATCH] * n_pages)
    return idx


def oracle_topk_check(idx, packed_bf16, q_host, n_queries, k, n_pages=512):
    """Top-k of `idx` (any dtype) restricted to its first n_pages pages vs the oracle of that dtype on the same rows."""
    import numpy as np
    import torch

    from oracle import maxsim_oracle as orc

    set_cpu_threads()
    rows = packed_bf16[: n_pages * P_PATCH * 256].view(torch.bfloat16).view(-1, DIM).float().cpu().numpy()
    off = orc.page_offsets([P_PATCH] * n_pages)
    allowed = np.zeros(idx.n_pages, dtype=bool)
    allowed[:n_pages] = True
    mask = idx.mask_from_pages(allowed)
    queries = [q_host[i * T_TOK:(i + 1) * T_TOK].numpy() for i in range(n_queries)]
    ts, ti, tc = idx.search_host(queries, k, allow_mask=mask)
    same, err = 0, 0.0
    for i, q in enumerate(queries):
        if idx.dtype_name == "bf16":
            want = orc.float_maxsim_c(orc.bf16_round_np(q), rows, off).astype(np.float64)
        elif idx.dtype_name == "int8":
            want = orc.int8_maxsim_c(orc.quantize_int8_np(q, idx.i8_scale), orc.quantize_int8_np(rows, idx.i8_scale), off) * idx.score_scale
        elif idx.dtype_name == "fp8":
            want = orc.float_maxsim_c(orc.dequantize_e4m3_np(orc.quantize_e4m3_np(q, idx.i8_scale)),
                                      orc.dequantize_e4m3_np(orc.quantize_e4m3_np(rows, idx.i8_scale)), off).astype(np.float64) * idx.score_scale
        else:
            want = orc.binary_maxsim_c(orc.sign_pack_c(q), orc.sign_pack_c(rows), off)[0]
        ws, wi = orc.topk_np(want, k)
        same += int(ti[i].tolist() == wi.tolist())
        err = max(err, float(np.max(np.abs(ts[i] - ws) / np.maximum(np.abs(ws), 1e-6))))
    exact = idx.dtype_name in ("int8", "binary")
    return {"id_lists_identical": f"{same}/{n_queries}", "max_rel_score_err": err, "tolerance": 0.0 if exact else 1e-3,
            "sample": f"first {n_pages} pages, {n_queries} queries, top-{k}"}


def time_search(idx, q_dev, q_lens, k, steps, warmup):
    """(step ms, scoring-kernel ms) of idx.search_device over `steps` calls, CUDA events."""
    import torch

    n_q = len(q_lens)
    out = (torch.empty((n_q, k), dtype=torch.float32, device=idx.device), torch.empty((n_q, k), dtype=torch.int64, device=idx.device),
           torch.empty((n_q,), dtype=torch.int32, device=idx.device))
    for _ in range(warmup):
        idx.search_device(q_dev, q_lens, k, out=out)
    torch.cuda.synchronize(idx.device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        idx.search_device(q_dev, q_lens, k, out=out)
    e1.record()
    torch.cuda.synchronize(idx.device)
    sm = idx.score_times_ms(min(steps, 256))
    return e0.elapsed_time(e1) / steps, sum(sm) / len(sm)


# ------------------------------------------------------------------------------------------------ the GPU arm
def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from morphik_core_b200.index import MaxSimIndex
    from morphik_core_b200.sharded import ShardedMaxSim

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the ONE JSON line: with NCCL_DEBUG=VERSION or WARN (set by some images) NCCL prints
        # "NCCL version ..." on stdout at communicator creation; unset it unless the user asked for INFO/TRACE
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")
        dist.init_process_group("nccl", device_id=device)
    peaks = load_peaks()
    n_q, k = args.bq, args.k
    free_b, total_b = torch.cuda.mem_get_info(device)
    n_pages = args.pages
    budget_pages = int((free_b - (24 << 30)) // (P_PATCH * 256))  # leave 24 GB for scratch, sub-shards and the FDE matrix
    if n_pages > budget_pages:  # a smaller shard would be a different workload with different inputs: say so instead
        raise SystemExit(f"--pages {n_pages} does not fit in the {free_b / 2**30:.1f} GiB free on cuda:{local_rank} "
                         f"(24 GiB stay free for the other legs): pass --pages {max(4096, budget_pages // 4096 * 4096)} or fewer")
    rows = n_pages * P_PATCH
    t_build0 = time.perf_counter()

    q_host = make_queries(n_q)  # identical on every rank
    anchors = topic_anchors(device)
    topic_pages = min(args.topic_pages, n_pages // 2)
    packed, planted = build_shard(n_pages, device, seed=1234 + rank, q_host=q_host, topic_pages=topic_pages, anchors=anchors)
    idx = MaxSimIndex(device=local_rank, dtype="bf16")
    idx.adopt_packed(packed, [P_PATCH] * n_pages)
    id_base = rank * n_pages
    sharded = ShardedMaxSim.from_index(idx, id_base=id_base) if world > 1 else None
    q_lens = [T_TOK] * n_q
    q_dev = q_host.to(device)
    q_pin = q_host.pin_memory()

    def dev_out(nq, kk=k):
        return (torch.empty((nq, kk), dtype=torch.float32, device=device), torch.empty((nq, kk), dtype=torch.int64, device=device),
                torch.empty((nq,), dtype=torch.int32, device=device))

    def pin_out(nq, kk=k):
        return (torch.empty((nq, kk), dtype=torch.float32).pin_memory(), torch.empty((nq, kk), dtype=torch.int64).pin_memory(),
                torch.empty((nq,), dtype=torch.int32).pin_memory())

    out_dev = [dev_out(n_q), dev_out(n_q)]
    out_pin = [pin_out(n_q), pin_out(n_q)]
    build_s = time.perf_counter() - t_build0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def run_device_steps(nsteps, qd=q_dev, lens=q_lens, outs=out_dev):
        """N = 1: b200ms_search_device; N > 1: the two-slot pipeline (begin i, then end i-1)."""
        if world == 1:
            for _ in range(nsteps):
                idx.search_device(qd, lens, k, out=outs[0])
            return
        prev = None
        for i in range(nsteps):
            t, _ = sharded.begin(qd, lens, k, out=outs[i & 1])
            if prev is not None:
                sharded.end(prev)
            prev = t
        sharded.end(prev)

    def run_e2e_steps(nsteps):
        if world == 1:
            for _ in range(nsteps):
                idx.search_host_flat(q_pin, q_lens, k, *out_pin[0])
            return
        prev = None
        for i in range(nsteps):
            t = idx.sharded_search_host_begin(q_pin, q_lens, k, id_base)
            if prev is not None:
                idx.sharded_search_host_end(prev, *out_pin[(i - 1) & 1])
            prev = t
        idx.sharded_search_host_end(prev, *out_pin[(nsteps - 1) & 1])

    # ---- correctness guard before timing: planted pages on top; at N > 1 identical lists on every rank + oracle on a sample
    run_device_steps(2)
    torch.cuda.synchronize(device)
    last = out_dev[1] if world > 1 else out_dev[0]
    top_ids = last[1].cpu()
    top1 = top_ids[:, 0].tolist()
    mine = sum(1 for qi in range(n_q) if rank * n_pages <= top1[qi] < (rank + 1) * n_pages and top1[qi] - id_base in planted[qi])
    multi_gpu_check = None
    if world == 1:
        assert mine >= n_q - 1, f"planted pages not retrieved ({mine}/{n_q}): the timed path is not computing MaxSim"
    else:
        hits = torch.tensor([mine], dtype=torch.int64, device=device)
        dist.all_reduce(hits)
        chk = torch.stack([last[1].double().sum(), (last[1].double() * torch.arange(1, k + 1, device=device)).sum(),
                           last[0].double().sum()])
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        identical = bool(torch.equal(lo, hi))
        assert identical, "merged top-k lists differ between ranks"
        assert int(hits.item()) >= n_q - 1, f"planted pages not retrieved across ranks ({int(hits.item())}/{n_q})"
        multi_gpu_check = {"merged_lists_identical_on_all_ranks": identical, "planted_top1_found": f"{int(hits.item())}/{n_q}"}
        # sharded search over a gathered sample vs the oracle: every rank contributes its first S pages
        S = args.check_pages
        sub = MaxSimIndex(device=local_rank, dtype="bf16")
        sub.adopt_packed(packed[: S * P_PATCH * 256], [P_PATCH] * S)
        sub_sh = ShardedMaxSim.from_index(sub, id_base=rank * S)
        nq_c = min(n_q, 4)
        cs, ci, cc = sub_sh.search(q_dev[: nq_c * T_TOK].contiguous(), [T_TOK] * nq_c, k)
        mine_rows = packed[: S * P_PATCH * 256].view(torch.bfloat16).view(S * P_PATCH, DIM)
        gathered = [torch.empty_like(mine_rows) for _ in range(world)] if rank == 0 else None
        dist.gather(mine_rows.contiguous(), gathered, dst=0)
        ok = torch.ones(1, dtype=torch.int64, device=device)
        if rank == 0:
            from oracle import maxsim_oracle as orc

            set_cpu_threads()
            all_rows = torch.cat(gathered).float().cpu().numpy()
            off = orc.page_offsets([P_PATCH] * (S * world))
            same, err = 0, 0.0
            for i in range(nq_c):
                want = orc.float_maxsim_c(orc.bf16_round_np(q_host[i * T_TOK:(i + 1) * T_TOK].numpy()), all_rows, off)
                ws, wi = orc.topk_np(want, k)
                same += int(ci[i].cpu().tolist() == wi.tolist())
                err = max(err, float(np.max(np.abs(cs[i].cpu().numpy() - ws) / np.maximum(np.abs(ws), 1e-6))))
            multi_gpu_check["oracle_on_gathered_sample"] = {
                "sample": f"first {S} pages of every rank = {S * world} pages, {nq_c} queries, top-{k}, sharded search vs oracle",
                "id_lists_identical": f"{same}/{nq_c}", "max_rel_score_err": err, "tolerance": 1e-3}
            ok[0] = int(same == nq_c and err <= 1e-3)
            del gathered, all_rows
        dist.broadcast(ok, src=0)
        assert int(ok.item()) == 1, "sharded search over the gathered sample disagrees with the oracle"
        sub.close()

    # ---- optional speed-proportional placement: shard sizes follow each GPU's measured scan rate (it differs under the
    #      1 kW power cap); pages_r are taken from the front of every rank's shard, the rest stays resident but unattached
    placement = {"mode": "equal", "pages_per_rank": [n_pages] * world}
    if world > 1 and args.placement == "speed":
        run_device_steps(max(6, args.warmup))
        torch.cuda.synchronize(device)
        sm = idx.score_times_ms(4)
        rate = torch.tensor([rows / (sum(sm) / len(sm))], dtype=torch.float64, device=device)
        rates = [torch.zeros_like(rate) for _ in range(world)]
        dist.all_gather(rates, rate)
        rates = [float(r.item()) for r in rates]
        mine_pages = int(n_pages * rates[rank] / max(rates)) // 1024 * 1024
        idx.adopt_packed(packed[: mine_pages * P_PATCH * 256], [P_PATCH] * mine_pages)
        pp = torch.tensor([mine_pages], dtype=torch.int64, device=device)
        allp = [torch.zeros_like(pp) for _ in range(world)]
        dist.all_gather(allp, pp)
        placement = {"mode": "speed-proportional (per-rank scan rates measured in warm-up)",
                     "pages_per_rank": [int(x.item()) for x in allp], "relative_rate": [r / max(rates) for r in rates]}
    total_rows = sum(placement["pages_per_rank"]) * P_PATCH

    # ---- value: device-resident inputs, CUDA events, max over ranks
    run_device_steps(max(args.warmup, args.settle_steps))  # warm-up (>= W): also lets the power-capped clocks settle
    barrier()
    launches0 = idx.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    ev0.record()
    run_device_steps(args.steps)
    ev1.record()
    barrier()
    t_host1 = time.perf_counter()
    clocks = sampler.stop(t_host0, t_host1)
    ms_total = ev0.elapsed_time(ev1)
    launches = idx.launch_count() - launches0
    # what a caller of the timed path receives from its last step (identical on every rank at N > 1)
    last_out = out_dev[(args.steps - 1) & 1] if world > 1 else out_dev[0]
    timed_outputs = {"topk_scores": last_out[0].cpu().numpy(), "topk_ids": last_out[1].cpu().numpy(),
                     "topk_counts": last_out[2].cpu().numpy()} if args.dump_outputs and rank == 0 else None
    score_ms = idx.score_times_ms(min(args.steps, 256))  # scoring kernels only, events recorded inside the timed region
    score_ms_avg = sum(score_ms) / len(score_ms)
    per_rank = None
    if world > 1:
        mine_t = torch.tensor([ms_total / args.steps, score_ms_avg, float(clocks["sm_mhz"] or 0), float(clocks["sm_mhz_min"] or 0)],
                              dtype=torch.float64, device=device)
        allt = [torch.zeros_like(mine_t) for _ in range(world)]
        dist.all_gather(allt, mine_t)
        allt = torch.stack(allt).cpu().numpy()
        ms_total = float(allt[:, 0].max()) * args.steps
        per_rank = {"step_ms": [round(float(x), 3) for x in allt[:, 0]], "scoring_kernel_ms": [round(float(x), 3) for x in allt[:, 1]],
                    "sm_mhz_median": [float(x) for x in allt[:, 2]], "sm_mhz_min": [float(x) for x in allt[:, 3]],
                    "scoring_kernel_ms_min_median_max": [float(np.min(allt[:, 1])), float(np.median(allt[:, 1])), float(np.max(allt[:, 1]))],
                    "limiter": "the slowest rank's scan (SM clock under the 1 kW power cap); the exchange is off the scan's stream"}
    ms_per_step = ms_total / args.steps
    value = total_rows / (ms_per_step * 1e-3)

    # ---- e2e: host buffers through the public C-ABI call, host<->device copies inside the timed region
    run_e2e_steps(args.warmup)
    barrier()
    t0 = time.perf_counter()
    run_e2e_steps(args.steps)
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = total_rows * args.steps / float(t.item())
    h2d = n_q * T_TOK * DIM * 4
    d2h = n_q * k * 12 + n_q * 4
    e2e_top1 = out_pin[(args.steps - 1) & 1][1][:, 0].tolist() if world > 1 else out_pin[0][1][:, 0].tolist()
    assert e2e_top1 == top1 or placement["mode"] != "equal", "e2e path returned a different top-1 than the device path"

    # ---- roofline of the dominant kernel (tensor-bound at 1024 resident query tokens)
    my_rows = placement["pages_per_rank"][rank] * P_PATCH
    flops_per_step = 2.0 * my_rows * DIM * n_q * T_TOK
    achieved_tf = flops_per_step / (score_ms_avg * 1e-3) / 1e12
    n_mtiles = (n_q * T_TOK + 127) // 128
    passes = (n_mtiles + 7) // 8
    tr = load_traffic()
    tkey = "maxsim_umma_pair<bf16,NM=4>"
    traffic_bytes = tr[tkey]["dram_bytes_per_patch_vector"] * my_rows if tr and tkey in tr else None
    roofline = {
        "kernel": "maxsim_umma_pair_kernel<bf16,NM=4>", "bound": "tensor", "achieved": achieved_tf,
        "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": achieved_tf / peaks["tflops_sustained"],
        "peak_kind": f"{peaks['source']} cuBLAS bf16 sustained (burst {peaks['tflops_burst']})",
        "frac_of_burst": achieved_tf / peaks["tflops_burst"], "traffic": traffic_bytes,
        "traffic_source": tr[tkey]["source"] if tr and tkey in tr else None,
        "launches_per_step": passes, "avg_launch_ms": score_ms_avg / passes, "score_ms_per_step": score_ms_avg,
        "algorithmic_flops_per_launch": flops_per_step / passes,
        "hbm_gbs_in_this_regime": passes * my_rows * DIM * 2 / (score_ms_avg * 1e-3) / 1e9,
    }

    # ---- the HBM-bound regime: one 32-token query over the same shard (every rank, local scan)
    q1 = q_dev[:T_TOK].contiguous()
    step1, sm1 = time_search(idx, q1, [T_TOK], k, args.steps, args.warmup)
    gbs = my_rows * DIM * 2 / (sm1 * 1e-3) / 1e9
    hbm = {"workload": f"same shard, ONE query x {T_TOK} tokens (B_q*T = 32: HBM-bound regime)", "bound": "hbm",
           "kernel": "maxsim_rowm_kernel<bf16,NG=1> (patch rows = MMA M operand, query tokens = N)", "achieved": gbs,
           "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
           "peak_kind": f"{peaks['source']} copy bandwidth (read+write; a read-only stream can exceed it)",
           "frac_of_nominal_7700_gbs": gbs / 7700.0,
           "patch_vectors_per_sec": my_rows / (sm1 * 1e-3), "score_ms": sm1, "step_ms": step1,
           "algorithmic_bytes_per_launch": my_rows * DIM * 2,
           "traffic": (tr["maxsim_rowm<bf16,NG=1>"]["dram_bytes_per_patch_vector"] * my_rows
                       if tr and "maxsim_rowm<bf16,NG=1>" in tr else None)}

    # ---- configs[3]: q-batch 256 (8192 query tokens = 8 CTA-pair passes) through the same (sharded) path
    cfg3 = None
    if not args.skip_legs:
        try:
            nq3 = 256
            q3_host = make_queries(nq3, seed=8642)
            q3 = q3_host.to(device)
            o3 = [dev_out(nq3), dev_out(nq3)]
            steps3 = max(2, min(args.steps, 4))
            run_device_steps(2, q3, [T_TOK] * nq3, o3)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_device_steps(steps3, q3, [T_TOK] * nq3, o3)
            e1.record()
            barrier()
            ms3 = e0.elapsed_time(e1) / steps3
            sm3 = idx.score_times_ms(steps3)
            sm3 = sum(sm3) / len(sm3)
            t3 = torch.tensor([ms3], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(t3, op=dist.ReduceOp.MAX)
            tf3 = 2.0 * my_rows * DIM * nq3 * T_TOK / (sm3 * 1e-3) / 1e12
            ids3 = o3[(steps3 - 1) & 1 if world > 1 else 0][1]
            # consistency: the first 32 queries of the batch-256 search must reproduce a batch-32 search of the same queries
            o32 = [dev_out(n_q), dev_out(n_q)]
            run_device_steps(1, q3[: n_q * T_TOK].contiguous(), q_lens, o32)
            torch.cuda.synchronize(device)
            same3 = bool(torch.equal(ids3[:n_q], o32[0][1]))
            cfg3 = {"workload": f"configs[3]: q-batch {nq3} x {T_TOK} tokens = {nq3 * T_TOK} query tokens, {n_pages} pages/GPU x {world} GPU(s), "
                                "NCCL top-k all-gather" if world > 1 else f"configs[3] shape on one GPU: q-batch {nq3} x {T_TOK} tokens, {n_pages} pages",
                    "value": total_rows / (float(t3.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t3.item()), "steps": steps3,
                    "bound": "tensor", "achieved": tf3, "peak": peaks["tflops_sustained"], "frac": tf3 / peaks["tflops_sustained"],
                    "roofline_unit": "TFLOP/s per GPU (rank 0)", "score_ms_per_step": sm3, "passes": (nq3 * T_TOK // 128 + 7) // 8,
                    "page_scores_per_sec": total_rows / P_PATCH * nq3 / (float(t3.item()) * 1e-3),
                    "topk_match": {"first_32_queries_equal_batch32_search": same3}}
            del q3, o3, o32
        except Exception as e:  # noqa: BLE001  (an extra leg must never break the bench line)
            cfg3 = {"error": repr(e)[:300]}

    # ---- configs[2]: bytes-per-score sweep on a sub-shard (one query = HBM regime, batch 32 = tensor regime)
    sweep = None
    if not args.skip_legs and rank == 0:
        try:
            sp = min(args.sweep_pages, n_pages)
            sweep = {"workload": f"configs[2] shape on a resident sub-shard: {sp} pages x {P_PATCH} patches (10M pages of int8 = 1.3 TB "
                                 "exceed one B200), one 32-token query (HBM-bound) and batch-32 (tensor-bound)", "points": {}}
            qb = q_dev
            for name in ("bf16", "int8", "fp8", "binary"):
                if name == "bf16":
                    sub = MaxSimIndex(device=local_rank, dtype="bf16")
                    sub.adopt_packed(packed[: sp * P_PATCH * 256], [P_PATCH] * sp)
                else:
                    sub = quantised_subshard(packed, sp, name, local_rank)
                rb = sub.row_bytes
                _, s1 = time_search(sub, q1, [T_TOK], k, max(10, args.steps), 3)
                _, s32 = time_search(sub, qb, q_lens, k, max(5, args.steps // 2), 2)
                g1 = sp * P_PATCH * rb / (s1 * 1e-3) / 1e9
                ops32 = 2.0 * sp * P_PATCH * DIM * n_q * T_TOK / (s32 * 1e-3) / 1e12
                pt = {"bytes_per_patch_vector": rb, "one_query": {"score_ms": s1, "achieved": g1, "unit": "GB/s", "peak": peaks["hbm_gbs"],
                                                                   "frac": g1 / peaks["hbm_gbs"], "frac_of_nominal_7700_gbs": g1 / 7700.0,
                                                                   "bound": "hbm" if name != "binary" else "instruction issue (bit expansion + epilogue), not hbm",
                                                                   "kernel": "maxsim_rowm_kernel",
                                                                   "patch_vectors_per_sec": sp * P_PATCH / (s1 * 1e-3)},
                      "batch32": {"score_ms": s32, "achieved": ops32, "unit": "TFLOP/s" if name in ("bf16", "fp8") else "TOP/s",
                                  "patch_vectors_per_sec": sp * P_PATCH / (s32 * 1e-3)}}
                if not args.no_cpu_baseline:
                    pt["topk_match"] = oracle_topk_check(sub, packed, q_host, 4, k)
                sweep["points"][name] = pt
                sub.close()
                del sub
                torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            sweep = {"error": repr(e)[:300]}

    # ---- configs[4]: FDE candidate generation + MaxSim rerank top-1000, p50 / p95 latency and recall on the topic pages
    two_stage = None
    if not args.skip_legs:
        try:
            two_stage = two_stage_leg(args, idx, packed, n_pages, topic_pages, anchors, sharded, world, rank, device, dist, k)
        except Exception as e:  # noqa: BLE001
            two_stage = {"error": repr(e)[:300]}
            if world > 1:
                raise

    # ---- configs[0], the reference's own CPU-runnable case (100 pages, one 32-token query): single-call latency through the
    #      C-ABI with host buffers, next to the reference formulation on the host CPU for the same shapes
    cfg0 = None
    if rank == 0 and world == 1:
        try:
            cfg0 = config0_latency(packed, q_pin, out_pin[0], k, args.no_cpu_baseline)
        except Exception as e:  # noqa: BLE001
            cfg0 = {"error": repr(e)[:200]}

    # ---- the reference's own GPU formulation on the same GPU (rank 0, N=1 only)
    torch_gpu = None
    if rank == 0 and world == 1:
        try:
            torch_gpu = torch_gpu_reference_rate(packed.view(torch.bfloat16).view(-1, DIM), q_dev, n_q)
        except Exception as e:  # noqa: BLE001
            torch_gpu = {"error": repr(e)[:200]}

    # ---- CPU baseline beside it (rank 0, N=1 only): the reference formulation on the first pages of the SAME shard; its
    #      scores are the oracle of topk_match (all queries)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cp = args.cpu_pages
        pages_np = packed[: cp * P_PATCH * 256].view(torch.bfloat16).view(cp, P_PATCH, DIM).float().cpu().numpy()
        from oracle import maxsim_oracle as orc

        qn = orc.bf16_round_np(q_host.numpy()).reshape(n_q, T_TOK, DIM)
        r = cpu_reference_rate(n_q, budget_s=args.cpu_budget, pages_np=pages_np, q_np=qn)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port", "host_cpus": os.cpu_count(),
               "sample": f"first {r['pages']} pages of the GPU shard x {P_PATCH} patches x {DIM}-d, {n_q} queries x {T_TOK} tokens, "
                         f"{r['seconds']:.1f} s of score_multi_vector (torch einsum, fp32) on the host"}
        try:
            cpu["topk_match"] = topk_match_from_scores(packed, q_pin, n_q, k, r["scores"], cp)
        except Exception as e:  # noqa: BLE001
            cpu["topk_match"] = {"error": repr(e)[:200]}
        del pages_np

    if timed_outputs is not None:
        dump_outputs(args.dump_outputs, timed_outputs)
    if rank == 0:
        cfg = workload_config(args, n_pages)
        cfg["placement"] = placement
        cfg["build_seconds"] = round(build_s, 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": cfg,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "b200ms_search_host (C-ABI, pinned host buffers, synchronous per call)" if world == 1 else
                           "b200ms_sharded_search_host_begin/_end (C-ABI: pinned H2D + scan + top-k + ncclAllGather + merge + D2H, two steps in flight)"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "hbm_regime": hbm, "cpu_baseline": cpu,
            "per_rank": per_rank, "multi_gpu_check": multi_gpu_check,
            "config2_sweep": sweep, "config3_bq256": cfg3, "config4_two_stage": two_stage,
            "torch_gpu_reference_formulation": torch_gpu, "config0_latency": cfg0,
            "page_scores_per_sec": value / P_PATCH * n_q, "top1_sample": top1[:4],
            "parity": {"bf16": "oracle pinned to the transformers port of score_multi_vector (tests/golden)", "int8": "no reference (new); oracle-defined",
                       "fp8": "no reference (new); oracle-defined", "binary": "SQL max_sim restated; pinned by 3 derived known answers only",
                       "fde": "UNPINNED (extension sources absent from the reference)"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def two_stage_leg(args, idx, packed, n_pages, topic_pages, anchors, sharded, world, rank, device, dist, k):
    """configs[4]: per-rank FDE matrix over the first `fde_pages` pages (built from the packed rows, time-boxed), single-query
    two-stage searches (FDE scan on tcgen05 -> top-1000 -> batched MaxSim rerank) with the one all-gather at N > 1; p50 / p95
    over `--latency-queries` topic queries; recall@{75,1000} of the exhaustive MaxSim top-10 on the topic pages."""
    import numpy as np
    import torch

    from morphik_core_b200.fde import TwoStageIndex
    from morphik_core_b200.index import MaxSimIndex
    from morphik_core_b200.sharded import exchange_bytes, exchange_views

    fp = min(args.fde_pages, n_pages)
    sub = MaxSimIndex(device=device.index, dtype="bf16")
    sub.adopt_packed(packed[: fp * P_PATCH * 256], [P_PATCH] * fp)
    two = TwoStageIndex(index=sub)
    t0 = time.perf_counter()
    two.rebuild_from_index()
    torch.cuda.synchronize(device)
    build_s = time.perf_counter() - t0
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=device)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(sub.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, src=0)
        sub.comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world)
    nlq = args.latency_queries
    tq_host, topics = make_topic_queries(nlq, anchors)
    tq = tq_host.to(device)
    id_base = rank * fp
    n_cand = 1000

    def one(qi, cands):
        """One single-query two-stage search; returns (scores, ids) on the device (merged across ranks at N > 1)."""
        q = tq[qi * T_TOK:(qi + 1) * T_TOK]
        ts, ti, tc, ev = two.search_device([q], k, cands, None, id_base)
        if world == 1:
            return ts, ti, ev
        xchg = torch.empty(exchange_bytes(1, k), dtype=torch.uint8, device=device)
        iv, sv = exchange_views(xchg, 1, k)
        iv.fill_(-1)
        sv.fill_(float("-inf"))
        iv[:, : ti.shape[1]].copy_(ti)
        sv[:, : ts.shape[1]].copy_(ts)
        ms, mi, mc = sub.allgather_topk(xchg, 1, k)
        return ms, mi, ev

    for qi in range(min(5, nlq)):
        one(qi, n_cand)
    torch.cuda.synchronize(device)
    lat, enc, scan, rer = [], [], [], []
    for qi in range(nlq):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        s, i, ev = one(qi, n_cand)
        _ = i.cpu()  # the caller reads its result
        lat.append((time.perf_counter() - t0) * 1e3)
        enc.append(ev[0].elapsed_time(ev[1]))
        scan.append(ev[1].elapsed_time(ev[2]))
        rer.append(ev[2].elapsed_time(ev[3]))
    lat_t = torch.tensor(lat, dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(lat_t, op=dist.ReduceOp.MAX)  # a query is done when its slowest rank is
    lat = np.sort(lat_t.cpu().numpy())
    # recall on the topic pages: exhaustive top-10 (masked to the topic pages) vs the two-stage answer with the same mask
    rec = {}
    tp = min(topic_pages, fp)
    if tp >= 1024:
        allowed = np.zeros(fp, dtype=bool)
        allowed[:tp] = True
        mask_np = sub.mask_from_pages(allowed)
        mask_dev = torch.from_numpy(mask_np.view(np.int32)).to(device)
        nrq = min(nlq, 32)
        queries = [tq_host[i * T_TOK:(i + 1) * T_TOK].numpy() for i in range(nrq)]
        ex_s, ex_i, _ = sub.search_host(queries, k, allow_mask=mask_np)
        for cands in (75, 1000):
            hit = tot = top1 = 0
            for qi in range(nrq):
                ts, ti, tc, _ = two.search_device([tq[qi * T_TOK:(qi + 1) * T_TOK]], k, cands, mask_dev, 0)
                got = set(ti[0].cpu().tolist())
                hit += len(got & set(ex_i[qi].tolist()))
                tot += k
                top1 += int(ex_i[qi][0] in got)
            rec[f"recall_at_{k}_with_{cands}_candidates"] = hit / tot
            rec[f"top1_retained_with_{cands}_candidates"] = top1 / nrq
        rec["corpus"] = (f"{tp} topic pages per GPU ({N_TOPICS} topics x graded noise levels; queries = topic anchors + noise), "
                         f"{nrq} queries, exhaustive MaxSim over the same pages as ground truth, rank {rank} shard")
    fde_bytes = fp * two.fde_dim * 2
    scan_med = float(np.median(scan))
    out = {"workload": f"configs[4]: FDE (20 x 32 x 16 = {two.fde_dim}-d bf16) candidate scan over {fp} pages/GPU x {world} GPU(s) + "
                       f"MaxSim rerank of the top-{n_cand}, single {T_TOK}-token queries, top-{k}",
           "p50_ms": float(lat[len(lat) // 2]), "p95_ms": float(lat[int(len(lat) * 0.95)]), "queries": nlq,
           "stage_ms_p50": {"encode_query": float(np.median(enc)), "fde_scan_plus_topk": scan_med, "rerank_scoring": float(np.median(rer))},
           "fde_scan": {"bound": "hbm", "algorithmic_bytes": fde_bytes, "note": "stage time includes the candidate top-k; see profiles/ for the kernel alone",
                        "achieved_lower_bound_gbs": fde_bytes / (scan_med * 1e-3) / 1e9},
           "fde_build": {"pages": fp, "seconds": build_s, "pages_per_s": fp / build_s},
           "recall": rec, "parity": "FDE unpinned (upstream sources absent); rerank scores are exact MaxSim"}
    # kernel-only scan rate for the roofline (1 query and 32 queries: the matrix is read once either way)
    qf1 = torch.randn((1, two.fde_dim), device=device)
    qf32 = torch.randn((32, two.fde_dim), device=device)
    for name, qf in (("scan_1_query", qf1), ("scan_32_queries", qf32)):
        for _ in range(3):
            two.fde_scores(qf)
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            two.fde_scores(qf)
        e1.record()
        torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / 10
        peaks = load_peaks()
        out["fde_scan"][name] = {"ms": ms, "achieved": fde_bytes / (ms * 1e-3) / 1e9, "unit": "GB/s", "peak": peaks["hbm_gbs"],
                                 "frac": fde_bytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "includes": "q hi/lo split + fde_scan_umma_kernel"}
    sub.close()
    return out


def dump_outputs(out_dir, arrays, limit_bytes=64 << 20):
    """Write each array as out_dir/<name>.npy: float32 / float64 as they are, integers as float64 (exact below 2^53)."""
    import numpy as np

    arrays = {name: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit_bytes:
        raise ValueError(f"{total} bytes of outputs exceed the {limit_bytes}-byte dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def main():
    import faulthandler

    wd = int(os.environ.get("B200MS_WATCHDOG_S", "0"))
    if wd > 0:  # multi-GPU runs under a lease: a hung collective dumps every thread's stack and exits instead of idling
        faulthandler.dump_traceback_later(wd, exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--pages", type=int, default=524288, help="pages per GPU in the resident shard")
    ap.add_argument("--bq", type=int, default=32, help="queries per batch")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--cpu-pages", type=int, default=4096, help="pages of the shard the CPU baseline / topk_match oracle scores")
    ap.add_argument("--ref-budget", type=float, default=6.0, help="seconds of CPU work per step of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-legs", action="store_true", help="only the headline numbers (value, e2e, roofline, hbm_regime)")
    ap.add_argument("--sweep-pages", type=int, default=65536, help="pages of the config-2 sweep sub-shard")
    ap.add_argument("--fde-pages", type=int, default=131072, help="pages per GPU in the config-4 two-stage index")
    ap.add_argument("--topic-pages", type=int, default=65536, help="leading pages of every shard that follow the topic model")
    ap.add_argument("--latency-queries", type=int, default=60)
    ap.add_argument("--check-pages", type=int, default=256, help="pages per rank in the multi-GPU oracle check")
    ap.add_argument("--settle-steps", type=int, default=12, help="untimed steps before the timed region (>= warmup): power-capped clocks settle")
    ap.add_argument("--placement", choices=["equal", "speed"], default=os.environ.get("B200MS_PLACEMENT", "equal"))
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the top-k of the last one (scores, ids, "
                    "counts) as DIR/<name>.npy, so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
