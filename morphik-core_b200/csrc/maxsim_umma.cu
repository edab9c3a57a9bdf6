// maxsim_umma.cu -- the float (bf16) and int8 MaxSim scorers on tcgen05 tensor cores.
//
// Replaces the reference's float scorer  einsum("bnd,csd->bcns").max(3).sum(2)  (colpali_engine
// score_multi_vector, called at core/vector_store/fast_multivector_store.py:553-555) and gives the new
// int8 variant (BASELINE config 3) the same structure.  The [B_q, C, T, P] similarity tensor is never
// materialised: each 128x128 (query tokens x patch rows) tile lives only in TMEM.
//
// Data layout in HBM
//   corpus rows   [n_rows, 128] bf16|s8, row-major, every page padded to a multiple of 32 rows ("chunks") by
//                 repeating its last row; chunk_page[c] = page index of chunk c
//   work units    unit_start[u] .. unit_start[u+1] = chunk range of unit u, always whole pages (so no page is
//                 ever split across CTAs and the per-token running max never crosses a CTA boundary)
//   queries       [n_groups*32, 128] same dtype, each query padded with zero rows to 32-row groups; an M tile is
//                 4 groups = 128 query tokens; TMEM lane i of the accumulator = query token i of the tile
//   scores        group_scores[g, p] (f32 | s32), g = 32-token group, p = page
//
// Kernels here: maxsim_umma_kernel<KIND,NM=1|2> (384 threads, two epilogue warpgroups) and maxsim_umma_w4_kernel<KIND,NM=4|8>
// (640 threads, four epilogue warpgroups).  The batch regime normally runs on CTA pairs (maxsim_umma_pair.cu); the round-1
// variants that lost their A/B (query operand from TMEM, replicated-query "split4" epilogue, two-warpgroup NM >= 4) are gone.
// KIND: 0 bf16, 1 int8, 2 fp8 e4m3 (umma_tile.cuh).
// Kernel (persistent, one CTA per SM, 384 threads, warp-specialised):
//   warp 0      TMA producer: streams 128-row patch tiles (SWIZZLE_128B boxes) through an S-stage mbarrier ring
//   warp 1      MMA issuer: for every patch tile and every resident query tile m < NM issues the K=128
//               contraction as 8 (bf16) / 4 (s8) tcgen05.mma 128x128xK into one of 4 TMEM accumulators
//   warp 2      TMEM allocator
//   warps 4-11  two epilogue warpgroups: tcgen05.ld the accumulator, per-thread max over the 32 columns of every
//               chunk (a thread owns one query token), fold into the running max of the current page, and at a
//               page boundary warp-shuffle-sum the 32 tokens of the group -> one score
// Roofline: HBM-bound while resident query tokens <= ~128-256 (B_q*T), tensor-bound above (SURVEY 8d).
// Algorithmic bytes per patch vector: 256 (bf16) / 128 (s8); flops per patch vector: 256 * query tokens.
#include "common.cuh"
#include "ptx.cuh"
#include "umma_tile.cuh"

namespace bms {

constexpr int kThreads = 384;

// TMA producer (one thread): the NM resident query tiles once, then every patch tile of this CTA's units through the
// num_stages ring.
template <int KIND, int NM>
__device__ __forceinline__ void produce_tiles(const CUtensorMap* tmap_rows, const CUtensorMap* tmap_q, const TileSmem& sm,
                                              int num_stages, const int32_t* __restrict__ unit_start,
                                              const int32_t* __restrict__ unit_end, int n_units, int m_tile_base) {
  using K = Kind<KIND>;
  const uint64_t pol_rows = policy_evict_first();
  const uint64_t pol_q = policy_evict_last();
  mbar_expect_tx(sm.qfull, NM * K::kTileBytes);
#pragma unroll
  for (int m = 0; m < NM; ++m)
#pragma unroll
    for (int p = 0; p < K::kPanels; ++p)
      tma_load_2d(tmap_q, sm.qfull, sm.q + m * K::kTileBytes + p * kSubtileBytes, p * K::kPanelElems,
                  (m_tile_base + m) * kTileM, pol_q);
  int stage = 0;
  uint32_t phase = 0;
  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
    const int n_tiles = (c1 - c0 + 3) >> 2;
    for (int t = 0; t < n_tiles; ++t) {
      mbar_wait(&sm.empty[stage], phase ^ 1);
      mbar_expect_tx(&sm.full[stage], K::kTileBytes);
      uint8_t* dst = sm.st + size_t(stage) * K::kTileBytes;
      const int row0 = (c0 + 4 * t) * kGroup;
#pragma unroll
      for (int p = 0; p < K::kPanels; ++p)
        tma_load_2d(tmap_rows, &sm.full[stage], dst + p * kSubtileBytes, p * K::kPanelElems, row0, pol_rows);
      if (++stage == num_stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  }
}

// One CTA per SM, NM = 1 or 2 resident query tiles, two epilogue warpgroups (warpgroup e owns query tiles m == e mod 2;
// at NM = 1 only warpgroup 0 works).  The lone-query / rerank kernel: HBM-bound while NM * 128 <= ~256 query tokens.
template <int KIND, int NM>
__global__ void __launch_bounds__(kThreads, 1)
maxsim_umma_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
                   const int32_t* __restrict__ chunk_page, const int32_t* __restrict__ unit_start,
                   const int32_t* __restrict__ unit_end, int slot_mode, int n_units, int m_tile_base, int n_groups_real,
                   const uint32_t* __restrict__ clamp_bits, typename Kind<KIND>::Acc* __restrict__ group_scores, int64_t ld,
                   int num_stages) {
  using K = Kind<KIND>;
  using Acc = typename K::Acc;
  static_assert(NM == 1 || NM == 2, "two-warpgroup form: 1 or 2 query tiles (4 and 8 run on maxsim_umma_w4_kernel)");

  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, NM * K::kTileBytes, K::kTileBytes, num_stages);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // tempty: one arrive per epilogue warp of the owning warpgroup
  const uint32_t tmem_base = tile_prologue<false>(sm, warp, &tmap_rows, &tmap_q, num_stages, 1, kNumAccum, 4);

  if (warp == 0) {
    if (lane == 0) produce_tiles<KIND, NM>(&tmap_rows, &tmap_q, sm, num_stages, unit_start, unit_end, n_units, m_tile_base);
  } else if (warp == 1) {
    // ================================================================ MMA issuer
    // The whole warp walks the loop (so every address/descriptor is warp-uniform and lives in uniform registers);
    // only the tcgen05.mma / tcgen05.commit themselves are issued by the lane elect.sync picks.
    constexpr uint32_t idesc = umma_idesc(KIND, kTileM, kTileN);
    constexpr uint32_t kTileDesc = K::kTileBytes >> 4;  // tile size in descriptor units (16 B)
    mbar_wait(sm.qfull, 0);
    tc_fence_after();
    const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.q));
    const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.st));
    int stage = 0;
    uint32_t phase = 0;
    uint32_t seq = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
      const int n_tiles = (c1 - c0 + 3) >> 2;
      for (int t = 0; t < n_tiles; ++t) {
        mbar_wait(&sm.full[stage], phase);
        tc_fence_after();
        const uint64_t bd = b_desc0 + uint64_t(uint32_t(stage) * kTileDesc);
#pragma unroll 1
        for (int m = 0; m < NM; ++m, ++seq) {
          const uint32_t buf = seq & (kNumAccum - 1);
          mbar_wait(&sm.tempty[buf], ((seq >> 2) & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            umma_tile<KIND>(tmem_base + buf * kTileN, a_desc0 + uint64_t(uint32_t(m) * kTileDesc), bd, idesc);
            umma_commit(&sm.tfull[buf]);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(&sm.empty[stage]);  // stage reusable once every query tile has consumed it
        __syncwarp();
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    // ================================================================ epilogue warpgroups
    const int wg = (warp - 4) >> 2;
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const uint32_t lane_base = tmem_base + (uint32_t(quad * 32) << 16);
    if (wg < NM) {
      const int m = wg;  // the query tile this warpgroup owns
      const int group = (m_tile_base + m) * 4 + quad;
      const bool active = group < n_groups_real;
      PageRun<Acc> run;
      uint32_t tile_seq = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
        const int n_tiles = (c1 - c0 + 3) >> 2;
        const auto emit = [&](int page, Acc rm) {
          store_group_score(group_scores, ld, group, slot_mode ? u : page, clamp_bits, rm);
        };
        for (int t = 0; t < n_tiles; ++t, ++tile_seq) {
          int pg[4];
          tile_pages(chunk_page, c0 + 4 * t, c1, pg);
          const uint32_t seq = tile_seq * NM + m;
          const uint32_t buf = seq & (kNumAccum - 1);
          const auto release = [&] { mbar_arrive(&sm.tempty[buf]); };  // accumulator drained: MMA may overwrite it
          mbar_wait(&sm.tfull[buf], (seq >> 2) & 1);
          tc_fence_after();
          if (active) {
            Acc cm[4];
            drain_accum(lane_base + buf * kTileN, cm, release);
            run.fold(pg, cm, emit);
          } else {
            release_accum(release);
          }
        }
        run.flush(emit);  // units end on a page boundary
      }
    }
  }
  tile_teardown<false>(warp, tmem_base);
}

// ================================================================================================================
// W4 form (NM = 4 for bf16, 4 or 8 for s8): FOUR epilogue warpgroups, warpgroup e owns TMEM accumulator e and the query
// tiles m with m % 4 == e.  In the two-warpgroup form each warpgroup needs ~820 of the 1024 cycles it has per accumulator
// (ncu: tensor pipe 73-76 % active although tcgen05.mma itself sustains 100 %, tools/umma_rate.cu); here every warpgroup
// has 2048 cycles per accumulator and five warps per SM sub-partition hide the TMEM-load latency.  640 threads.
constexpr int kThreadsW4 = 640;

template <int KIND, int NM>
__global__ void __launch_bounds__(kThreadsW4, 1)
maxsim_umma_w4_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
                      const int32_t* __restrict__ chunk_page, const int32_t* __restrict__ unit_start,
                      const int32_t* __restrict__ unit_end, int slot_mode, int n_units, int m_tile_base, int n_groups_real,
                      const uint32_t* __restrict__ clamp_bits, typename Kind<KIND>::Acc* __restrict__ group_scores, int64_t ld,
                      int num_stages) {
  using K = Kind<KIND>;
  using Acc = typename K::Acc;
  static_assert(NM % 4 == 0, "W4 form needs a multiple of four query tiles");
  constexpr int MPW = NM / 4;                  // query tiles per epilogue warpgroup

  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, NM * K::kTileBytes, K::kTileBytes, num_stages);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t tmem_base = tile_prologue<false>(sm, warp, &tmap_rows, &tmap_q, num_stages, 1, kNumAccum, 4);

  if (warp == 0) {
    if (lane == 0) produce_tiles<KIND, NM>(&tmap_rows, &tmap_q, sm, num_stages, unit_start, unit_end, n_units, m_tile_base);
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc(KIND, kTileM, kTileN);
    constexpr uint32_t kTileDesc = K::kTileBytes >> 4;
    mbar_wait(sm.qfull, 0);
    tc_fence_after();
    const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.q));
    const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.st));
    int stage = 0;
    uint32_t phase = 0;
    uint32_t use = 0;  // uses of every accumulator so far (each tile uses each buffer MPW times)
    for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
      const int n_tiles = (c1 - c0 + 3) >> 2;
      for (int t = 0; t < n_tiles; ++t) {
        mbar_wait(&sm.full[stage], phase);
        tc_fence_after();
        const uint64_t bd = b_desc0 + uint64_t(uint32_t(stage) * kTileDesc);
#pragma unroll 1
        for (int m = 0; m < NM; ++m) {
          const uint32_t buf = m & 3;
          const uint32_t n = use + (m >> 2);
          mbar_wait(&sm.tempty[buf], (n & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            umma_tile<KIND>(tmem_base + buf * kTileN, a_desc0 + uint64_t(uint32_t(m) * kTileDesc), bd, idesc);
            umma_commit(&sm.tfull[buf]);
          }
          __syncwarp();
        }
        use += MPW;
        if (elect_one()) umma_commit(&sm.empty[stage]);
        __syncwarp();
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    const int wg = (warp - 4) >> 2;  // 0..3 = accumulator buffer owned
    const int quad = warp & 3;
    const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + wg * kTileN;
    const auto release = [&] { mbar_arrive(&sm.tempty[wg]); };
    PageRun<Acc> run[MPW];
    uint32_t use = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
      const int n_tiles = (c1 - c0 + 3) >> 2;
      for (int t = 0; t < n_tiles; ++t) {
        int pg[4];
        tile_pages(chunk_page, c0 + 4 * t, c1, pg);
#pragma unroll
        for (int i = 0; i < MPW; ++i, ++use) {
          const int group = (m_tile_base + wg + 4 * i) * 4 + quad;
          mbar_wait(&sm.tfull[wg], use & 1);
          tc_fence_after();
          if (group < n_groups_real) {
            Acc cm[4];
            drain_accum(taddr, cm, release);
            run[i].fold(pg, cm, [&](int page, Acc rm) {
              store_group_score(group_scores, ld, group, slot_mode ? u : page, clamp_bits, rm);
            });
          } else {
            release_accum(release);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < MPW; ++i) {
        const int group = (m_tile_base + wg + 4 * i) * 4 + quad;
        run[i].flush([&](int page, Acc rm) {
          store_group_score(group_scores, ld, group, slot_mode ? u : page, clamp_bits, rm);
        });
      }
    }
  }
  tile_teardown<false>(warp, tmem_base);
}

// ---------------------------------------------------------------------------------------------- host side
// One launch of a one-CTA form: NM = 1 / 2 on maxsim_umma_kernel with up to 14 stages (16 KB tiles: 8 stages = 128 KB in
// flight left the one-byte scans latency-bound), NM = 4 / 8 on the W4 form with up to 8.
template <int KIND, int NM>
static int launch_one(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int m_tile_base, int n_groups_real,
                      void* scores, int64_t ld, cudaStream_t s) {
  using K = Kind<KIND>;
  const auto launch = [&](auto kern, const char* name, int threads, int max_stages) {
    return launch_persistent(h, kern, name, threads, NM * K::kTileBytes, K::kTileBytes, max_stages, up.n_units, s,
                             h->corpus.tmap, tq, static_cast<const int32_t*>(h->chunk_page.p), up.start, up.end,
                             up.slot_mode, up.n_units, m_tile_base, n_groups_real, up.clamp_bits,
                             static_cast<typename K::Acc*>(scores), ld);
  };
  if constexpr (NM <= 2) return launch(maxsim_umma_kernel<KIND, NM>, "maxsim_umma", kThreads, 14);
  else return launch(maxsim_umma_w4_kernel<KIND, NM>, "maxsim_umma_w4", kThreadsW4, 8);
}

// Pass planner: score query tiles [0, n_mtiles) against the unit plan with as few passes over the corpus as possible.
//   CTA-pair forms (maxsim_umma_pair.cu) hold 2*per query tiles per pass; pick the largest per whose phantom (zero) tiles
//   stay below a quarter of the pass -- 5 tiles run as 4 + 1, not as 8 (measured per pass at 32768 pages: 8 tiles 5.08 ms,
//   4 tiles ~2.5 ms, one tile 1.28 ms); pair_cta = 2 (default) also sends exactly two tiles to the two-tile pair kernel.
//   One-CTA forms: a single tile (the lone query, HBM-bound) always; 2 / 4 / 8 tiles only where CTA pairs cannot be
//   co-scheduled (pair_cta = 0 or a partition without whole TPCs) -- same results, bit for bit.
template <int KIND>
static int launch_kind(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int n_groups_real, int n_mtiles, void* scores,
                       int64_t ld, cudaStream_t s) {
  constexpr int kMaxNM = Kind<KIND>::kMaxNM;
  int base = 0;
  while (base < n_mtiles) {
    const int rem = n_mtiles - base;
    if (h->pair_cta && rem >= (h->pair_cta >= 2 ? 2 : 3)) {
      int per = kMaxNM;
      while (per > 1 && rem < 2 * per - (per >= 4 ? per / 4 : 1)) per >>= 1;
      if (per == 1 && (h->pair_cta < 2 || rem < 2)) per = 0;
      if (per > 0) {
        const int e2 = launch_score_umma_pair(h, up, tq, per, base, n_groups_real, scores, ld, s);
        if (e2 == B200MS_OK) {
          base += 2 * per;
          continue;
        }
        if (e2 != B200MS_EUNSUPPORTED_PAIR) return e2;
        h->pair_cta = 0;  // e.g. a partition without whole TPCs: the one-CTA kernels below do the same work
      }
    }
    int nm = 1;
    while (nm < rem && nm < kMaxNM) nm <<= 1;  // round up: a phantom (all-zero) tile beats a 2nd pass over the corpus
    int e;
    switch (nm) {
      case 1: e = launch_one<KIND, 1>(h, up, tq, base, n_groups_real, scores, ld, s); break;
      case 2: e = launch_one<KIND, 2>(h, up, tq, base, n_groups_real, scores, ld, s); break;
      case 4: e = launch_one<KIND, 4>(h, up, tq, base, n_groups_real, scores, ld, s); break;
      default:
        if constexpr (kMaxNM >= 8) {
          e = launch_one<KIND, 8>(h, up, tq, base, n_groups_real, scores, ld, s);
        } else {
          e = set_error(h, B200MS_EINVAL, "maxsim_umma: bad NM");
        }
    }
    if (e) return e;
    base += nm;
  }
  return B200MS_OK;
}

// m_tile >= 0: score only that query tile, on the single-tile kernel -- the batched rerank launches each query tile against
// its own (short) candidate lists.
int launch_score_umma(b200ms_t* h, const UnitPlan* plan, const void* q_packed, int n_groups_real, void* group_scores,
                      int64_t ld, cudaStream_t s, int m_tile) {
  const Corpus& c = h->corpus;
  UnitPlan up;
  if (plan) {
    up = *plan;
  } else {  // full scan: unit u = [unit_start[u], unit_start[u+1])
    up.start = static_cast<const int32_t*>(h->unit_start.p);
    up.end = up.start + 1;
    up.n_units = c.n_units;
    up.slot_mode = 0;
  }
  if (!c.has_tmap) return set_error(h, B200MS_ESTATE, "score: corpus has no TMA descriptor");
  const int n_groups_padded = (n_groups_real + 3) & ~3;
  const int n_mtiles = n_groups_padded / 4;
  const CUtensorMap* tq;
  if (int e = query_tmap(h, q_packed, c.dtype, n_groups_padded * kGroup, kTileM, &tq)) return e;
  if (m_tile >= 0) {
    switch (kind_of_dtype(c.dtype)) {
      case 0: return launch_one<0, 1>(h, up, *tq, m_tile, n_groups_real, group_scores, ld, s);
      case 1: return launch_one<1, 1>(h, up, *tq, m_tile, n_groups_real, group_scores, ld, s);
      default: return launch_one<2, 1>(h, up, *tq, m_tile, n_groups_real, group_scores, ld, s);
    }
  }
  switch (kind_of_dtype(c.dtype)) {
    case 0: return launch_kind<0>(h, up, *tq, n_groups_real, n_mtiles, group_scores, ld, s);
    case 1: return launch_kind<1>(h, up, *tq, n_groups_real, n_mtiles, group_scores, ld, s);
    case 2: return launch_kind<2>(h, up, *tq, n_groups_real, n_mtiles, group_scores, ld, s);
    default: return set_error(h, B200MS_ESTATE, "score: corpus dtype has no tcgen05 scorer");
  }
}

}  // namespace bms
