// maxsim_umma_pair.cu -- the batch (tensor-bound) regime of the bf16 / int8 MaxSim scorer on CTA PAIRS.
//
// Same contract, HBM layout and page logic as maxsim_umma.cu (which replaces colpali_engine's score_multi_vector,
// call site core/vector_store/fast_multivector_store.py:553-555); only the mapping onto the machine differs:
//
//   * a cluster of two CTAs (the two SMs of a TPC) issues tcgen05.mma.cta_group::2 with M = 256, N = 256:
//       A  = 256 query tokens, 128 resident in each CTA's shared memory (so one pair holds 2*NM query tiles)
//       B  = 256 patch rows, 128 in each CTA's shared memory.  The two halves are INDEPENDENT streams of work units:
//            the leader CTA streams units blockIdx.x, +gridDim.x, ... and the peer its own list, so accumulator columns
//            [0,128) hold pages of the leader's stream and [128,256) pages of the peer's -- no page is ever split
//            between the halves and the epilogue needs no cross-half combine.
//     Per 128x256x16 MMA step each SM reads 4 KB of A and 4 KB of B from shared memory in 128 cycles (64 B/clk)
//     where the one-CTA form (128x128x16 in 64 cycles) needs 128 B/clk -- the whole shared-memory bandwidth -- and
//     every patch row is fetched from HBM/L2 once per 2*NM query tiles instead of once per NM.
//   * TMEM: two accumulators of 256 fp32/s32 columns in each CTA (its 128 tokens x 256 patch rows).
//   * warps (640 threads per CTA): 0 TMA producer of this CTA's stream, 1 MMA issuer (leader only), 2 TMEM allocator,
//     4-19 four epilogue warpgroups: warpgroup e drains accumulator e>>1, column half e&1 (= stream e&1), i.e. the query
//     tiles m with m % 2 == e>>1 -- exactly the W4 epilogue of maxsim_umma.cu per (accumulator, half).
//   * barriers: full[s] lives in the leader (both producers' TMA bytes land on it), empty[s] / tfull[b] are arrived in
//     both CTAs by multicast tcgen05.commit, tempty[b] lives in the leader and collects 16 warp arrivals (8 remote).
// Used for passes of >= 2 query tiles (> 128 query tokens; the two-tile form is maxsim_umma_pair1_kernel below); a single
// tile (<= 128 tokens, the lone-query case) is HBM-bound and stays on maxsim_umma.cu.  Pass planning: launch_kind().
#include "common.cuh"
#include "ptx.cuh"
#include "umma_tile.cuh"

namespace bms {

constexpr int kThreadsPair = 640;
constexpr int kPairN = 2 * kTileN;  // accumulator columns: 128 patch rows of each stream

template <int KIND, int NM>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsPair, 1)
maxsim_umma_pair_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
                        const int32_t* __restrict__ chunk_page, const int32_t* __restrict__ unit_start,
                        const int32_t* __restrict__ unit_end, int slot_mode, int n_units, int m_tile_base,
                        int n_groups_real, const uint32_t* __restrict__ clamp_bits,
                        typename Kind<KIND>::Acc* __restrict__ group_scores, int64_t ld, int num_stages) {
  using K = Kind<KIND>;
  using Acc = typename K::Acc;
  static_assert(NM % 2 == 0, "pair form: an even number of query tiles per CTA (tile m uses accumulator m & 1)");
  constexpr int MPW = NM / 2;  // query tiles per epilogue warpgroup

  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, NM * K::kTileBytes, K::kTileBytes, num_stages);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();           // 0 = leader (issues the MMAs), 1 = peer
  const int stream0 = int(blockIdx.x) - int(rank);   // virtual CTA index of the leader's unit stream; the peer's is +1

  // Both streams advance in lock step (one 128-row tile each per iteration); the shorter one pads with dummy tiles.
  int n_iter = 0;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    int acc = 0;
    for (int u = stream0 + s + lane * int(gridDim.x); u < n_units; u += 32 * int(gridDim.x))
      acc += (__ldg(unit_end + u) - __ldg(unit_start + u) + 3) >> 2;
    n_iter = max(n_iter, warp_sum(acc));
  }

  // tempty: 2 CTAs x 2 warpgroups x 4 warps
  const uint32_t tmem_base = tile_prologue<true>(sm, warp, &tmap_rows, &tmap_q, num_stages, 1, 2, 16);

  if (warp == 0) {
    if (lane == 0) {
      const uint64_t pol_rows = policy_evict_first();
      const uint64_t pol_q = policy_evict_last();
      const uint32_t full_l = mapa_rank(smem_u32(sm.full), 0);   // the LEADER's barriers collect both CTAs' bytes
      const uint32_t qfull_l = mapa_rank(smem_u32(sm.qfull), 0);
      if (rank == 0) mbar_expect_tx(sm.qfull, 2 * NM * K::kTileBytes);
#pragma unroll
      for (int m = 0; m < NM; ++m)
#pragma unroll
        for (int p = 0; p < K::kPanels; ++p)
          tma_load_2d_pair(&tmap_q, qfull_l, sm.q + m * K::kTileBytes + p * kSubtileBytes, p * K::kPanelElems,
                           (m_tile_base + int(rank) * NM + m) * kTileM, pol_q);
      int stage = 0;
      uint32_t phase = 0;
      int k = 0;
      auto load_tile = [&](int row0) {
        mbar_wait(&sm.empty[stage], phase ^ 1);
        if (rank == 0) mbar_expect_tx(&sm.full[stage], 2 * K::kTileBytes);
        uint8_t* dst = sm.st + size_t(stage) * K::kTileBytes;
#pragma unroll
        for (int p = 0; p < K::kPanels; ++p)
          tma_load_2d_pair(&tmap_rows, full_l + uint32_t(stage) * 8u, dst + p * kSubtileBytes, p * K::kPanelElems, row0,
                           pol_rows);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      };
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
        const int n_tiles = (c1 - c0 + 3) >> 2;
        for (int t = 0; t < n_tiles; ++t, ++k) load_tile((c0 + 4 * t) * kGroup);
      }
      for (; k < n_iter; ++k) load_tile(0);  // this stream is exhausted: keep the pair in step
      // tail: the multicast commits of the last stages must land before this CTA may exit
      for (int i = 0; i < num_stages; ++i) {
        mbar_wait(&sm.empty[stage], phase ^ 1);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc(KIND, 2 * kTileM, kPairN);
      constexpr uint32_t kTileDesc = K::kTileBytes >> 4;
      mbar_wait(sm.qfull, 0);
      tc_fence_after();
      const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.q));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.st));
      int stage = 0;
      uint32_t phase = 0;
      uint32_t use = 0;  // uses of each accumulator so far
      for (int k = 0; k < n_iter; ++k) {
        mbar_wait(&sm.full[stage], phase);
        tc_fence_after();
        const uint64_t bd = b_desc0 + uint64_t(uint32_t(stage) * kTileDesc);
#pragma unroll 1
        for (int m = 0; m < NM; ++m) {
          const uint32_t buf = m & 1;
          const uint32_t n = use + (m >> 1);
          mbar_wait(&sm.tempty[buf], (n & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            umma_tile<KIND, true>(tmem_base + buf * kPairN, a_desc0 + uint64_t(uint32_t(m) * kTileDesc), bd, idesc);
            umma2_commit_mc(&sm.tfull[buf], 3);
          }
          __syncwarp();
        }
        use += MPW;
        if (elect_one()) umma2_commit_mc(&sm.empty[stage], 3);
        __syncwarp();
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    const int e = (warp - 4) >> 2;
    const int buf = e >> 1;  // accumulator drained by this warpgroup
    const int half = e & 1;  // column half = unit stream
    const int quad = warp & 3;
    const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + buf * kPairN + half * kTileN;
    const uint32_t tempty_l = mapa_rank(smem_u32(&sm.tempty[buf]), 0);
    const auto release = [&] { mbar_arrive_cluster(tempty_l); };
    PageRun<Acc> run[MPW];
    uint32_t use = 0;
    int k = 0;
    for (int u = stream0 + half; u < n_units; u += gridDim.x) {
      const int c0 = __ldg(unit_start + u), c1 = __ldg(unit_end + u);
      const int n_tiles = (c1 - c0 + 3) >> 2;
      for (int t = 0; t < n_tiles; ++t, ++k) {
        int pg[4];
        tile_pages(chunk_page, c0 + 4 * t, c1, pg);
#pragma unroll
        for (int i = 0; i < MPW; ++i, ++use) {
          const int group = (m_tile_base + int(rank) * NM + buf + 2 * i) * 4 + quad;
          mbar_wait(&sm.tfull[buf], use & 1);
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
        const int group = (m_tile_base + int(rank) * NM + buf + 2 * i) * 4 + quad;
        run[i].flush([&](int page, Acc rm) {
          store_group_score(group_scores, ld, group, slot_mode ? u : page, clamp_bits, rm);
        });
      }
    }
    for (; k < n_iter; ++k) {  // dummy tiles of an exhausted stream: keep the accumulator hand-shake going
#pragma unroll
      for (int i = 0; i < MPW; ++i, ++use) {
        mbar_wait(&sm.tfull[buf], use & 1);
        __syncwarp();
        if (lane == 0) release();
      }
    }
  }
  tile_teardown<true>(warp, tmem_base);
}

// ================================================================================================================
// Two-tile form (129..256 query tokens): ONE query tile per CTA, so a pair holds 2 tiles and every MMA batch fills a whole
// accumulator (tile k uses accumulator k & 1).  To keep "one epilogue warpgroup = one unit stream" each CTA now feeds TWO
// unit streams, alternating per iteration: even iterations carry a tile of its stream 2c, odd ones a tile of stream 2c+1
// (c = blockIdx.x; a stream walks units v, v + 2*gridDim.x, ...).  Warpgroup e drains accumulator e>>1 (= iteration parity)
// and column half e&1 (= the CTA that loaded those rows), i.e. exactly one of the pair's four streams.
template <int KIND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsPair, 1)
maxsim_umma_pair1_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
                         const int32_t* __restrict__ chunk_page, const int32_t* __restrict__ unit_start,
                         const int32_t* __restrict__ unit_end, int slot_mode, int n_units, int m_tile_base,
                         int n_groups_real, const uint32_t* __restrict__ clamp_bits,
                         typename Kind<KIND>::Acc* __restrict__ group_scores, int64_t ld, int num_stages) {
  using K = Kind<KIND>;
  using Acc = typename K::Acc;

  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, K::kTileBytes, K::kTileBytes, num_stages);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int stream0 = 2 * (int(blockIdx.x) - int(rank));  // first of the pair's four streams
  const int vstride = 2 * int(gridDim.x);

  // iterations per parity = the longest of the four streams (shorter ones pad with dummy tiles)
  int n_half = 0;
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    int acc = 0;
    for (int u = stream0 + s + lane * vstride; u < n_units; u += 32 * vstride)
      acc += (__ldg(unit_end + u) - __ldg(unit_start + u) + 3) >> 2;
    n_half = max(n_half, warp_sum(acc));
  }
  const int n_iter = 2 * n_half;

  const uint32_t tmem_base = tile_prologue<true>(sm, warp, &tmap_rows, &tmap_q, num_stages, 1, 2, 16);

  if (warp == 0) {
    if (lane == 0) {
      const uint64_t pol_rows = policy_evict_first();
      const uint64_t pol_q = policy_evict_last();
      const uint32_t full_l = mapa_rank(smem_u32(sm.full), 0);
      const uint32_t qfull_l = mapa_rank(smem_u32(sm.qfull), 0);
      if (rank == 0) mbar_expect_tx(sm.qfull, 2 * K::kTileBytes);
#pragma unroll
      for (int p = 0; p < K::kPanels; ++p)
        tma_load_2d_pair(&tmap_q, qfull_l, sm.q + p * kSubtileBytes, p * K::kPanelElems,
                         (m_tile_base + int(rank)) * kTileM, pol_q);
      UnitWalk w0, w1;
      w0.init(2 * int(blockIdx.x), vstride, unit_start, unit_end, n_units);
      w1.init(2 * int(blockIdx.x) + 1, vstride, unit_start, unit_end, n_units);
      int stage = 0;
      uint32_t phase = 0;
      for (int k = 0; k < n_iter; ++k) {
        int row0 = 0;  // dummy tile once this stream is exhausted
        if (k & 1) {
          if (w1.valid(n_units)) {
            row0 = w1.chunk() * kGroup;
            w1.next(unit_start, unit_end, n_units);
          }
        } else if (w0.valid(n_units)) {
          row0 = w0.chunk() * kGroup;
          w0.next(unit_start, unit_end, n_units);
        }
        mbar_wait(&sm.empty[stage], phase ^ 1);
        if (rank == 0) mbar_expect_tx(&sm.full[stage], 2 * K::kTileBytes);
        uint8_t* dst = sm.st + size_t(stage) * K::kTileBytes;
#pragma unroll
        for (int p = 0; p < K::kPanels; ++p)
          tma_load_2d_pair(&tmap_rows, full_l + uint32_t(stage) * 8u, dst + p * kSubtileBytes, p * K::kPanelElems, row0,
                           pol_rows);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      for (int i = 0; i < num_stages; ++i) {  // tail: let the last multicast commits land before this CTA may exit
        mbar_wait(&sm.empty[stage], phase ^ 1);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc(KIND, 2 * kTileM, kPairN);
      constexpr uint32_t kTileDesc = K::kTileBytes >> 4;
      mbar_wait(sm.qfull, 0);
      tc_fence_after();
      const uint64_t ad = umma_desc_kmajor_sw128(smem_u32(sm.q));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.st));
      int stage = 0;
      uint32_t phase = 0;
      for (int k = 0; k < n_iter; ++k) {
        const uint32_t buf = k & 1;
        mbar_wait(&sm.full[stage], phase);
        mbar_wait(&sm.tempty[buf], ((uint32_t(k) >> 1) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          umma_tile<KIND, true>(tmem_base + buf * kPairN, ad, b_desc0 + uint64_t(uint32_t(stage) * kTileDesc), idesc);
          umma2_commit_mc(&sm.tfull[buf], 3);
          umma2_commit_mc(&sm.empty[stage], 3);
        }
        __syncwarp();
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    const int e = (warp - 4) >> 2;
    const int buf = e >> 1;  // accumulator = iteration parity = stream parity
    const int half = e & 1;  // column half = CTA whose producer loaded these rows
    const int quad = warp & 3;
    const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + buf * kPairN + half * kTileN;
    const uint32_t tempty_l = mapa_rank(smem_u32(&sm.tempty[buf]), 0);
    const auto release = [&] { mbar_arrive_cluster(tempty_l); };
    const int group = (m_tile_base + int(rank)) * 4 + quad;
    UnitWalk w;
    w.init(stream0 + 2 * half + buf, vstride, unit_start, unit_end, n_units);
    PageRun<Acc> run;
    int last_u = -1;
    const auto emit = [&](int page, Acc rm) {
      store_group_score(group_scores, ld, group, slot_mode ? last_u : page, clamp_bits, rm);
    };
    for (int n = 0; n < n_half; ++n) {
      mbar_wait(&sm.tfull[buf], n & 1);
      tc_fence_after();
      if (group < n_groups_real && w.valid(n_units)) {
        if (w.u != last_u) {  // a new unit starts: units are whole pages
          run.flush(emit);
          last_u = w.u;
        }
        int pg[4];
        tile_pages(chunk_page, w.chunk(), w.c1, pg);
        Acc cm[4];
        drain_accum(taddr, cm, release);
        run.fold(pg, cm, emit);
        w.next(unit_start, unit_end, n_units);
      } else {
        release_accum(release);
      }
    }
    run.flush(emit);
  }
  tile_teardown<true>(warp, tmem_base);
}

// Once per handle: can this device co-schedule CTA pairs of this size at all?
static bool pairs_schedulable(b200ms_t* h, const void* kern, uint32_t smem) {
  if (h->pair_clusters < 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2);
    cfg.blockDim = dim3(kThreadsPair);
    cfg.dynamicSmemBytes = smem;
    int n = 0;
    const cudaError_t qe = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
    if (qe != cudaSuccess) (void)cudaGetLastError();
    h->pair_clusters = qe == cudaSuccess ? n : 0;
  }
  return h->pair_clusters >= 1;
}

// NM = query tiles per CTA: 1 on the two-tile kernel, 2 / 4 / 8 on maxsim_umma_pair_kernel.  B200MS_EUNSUPPORTED_PAIR:
// the device cannot co-schedule the pair, and the caller falls back to the one-CTA kernels (still CUDA).
template <int KIND, int NM>
static int launch_pair(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int m_tile_base, int n_groups_real,
                       void* scores, int64_t ld, cudaStream_t s) {
  using K = Kind<KIND>;
  const auto launch = [&](auto kern, const char* name, int want) {
    int stages;
    uint32_t smem;
    if (int e = size_stage_ring(h, reinterpret_cast<const void*>(kern), name, NM * K::kTileBytes, K::kTileBytes, 8, &stages,
                                &smem))
      return e;
    if (up.n_units < 1) return int(B200MS_OK);
    if (!pairs_schedulable(h, reinterpret_cast<const void*>(kern), smem)) return B200MS_EUNSUPPORTED_PAIR;
    int grid = (h->max_ctas > 0 ? h->max_ctas : h->num_sms) & ~1;  // whole pairs
    if (grid > want) grid = want;
    if (grid < 2) grid = 2;
    kern<<<grid, kThreadsPair, smem, s>>>(h->corpus.tmap, tq, static_cast<const int32_t*>(h->chunk_page.p), up.start, up.end,
                                         up.slot_mode, up.n_units, m_tile_base, n_groups_real, up.clamp_bits,
                                         static_cast<typename K::Acc*>(scores), ld, stages);
    h->launches++;
    return check_cuda(h, cudaGetLastError(), name);
  };
  if constexpr (NM == 1) {
    return launch(maxsim_umma_pair1_kernel<KIND>, "maxsim_umma_pair1", (((up.n_units + 1) / 2) + 1) & ~1);  // 2 streams per CTA
  } else {
    return launch(maxsim_umma_pair_kernel<KIND, NM>, "maxsim_umma_pair", (up.n_units + 1) & ~1);
  }
}

// nm = query tiles per CTA (1, 2, 4; 8 for the one-byte dtypes): one launch scores 2*nm query tiles [m_tile_base, m_tile_base + 2*nm).
template <int KIND>
static int launch_pair_kind(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int nm, int m_tile_base,
                            int n_groups_real, void* scores, int64_t ld, cudaStream_t s) {
  switch (nm) {
    case 1: return launch_pair<KIND, 1>(h, up, tq, m_tile_base, n_groups_real, scores, ld, s);
    case 2: return launch_pair<KIND, 2>(h, up, tq, m_tile_base, n_groups_real, scores, ld, s);
    case 4: return launch_pair<KIND, 4>(h, up, tq, m_tile_base, n_groups_real, scores, ld, s);
    case 8:
      if constexpr (Kind<KIND>::kMaxNM >= 8) return launch_pair<KIND, 8>(h, up, tq, m_tile_base, n_groups_real, scores, ld, s);
      [[fallthrough]];
    default:
      return set_error(h, B200MS_EINVAL, "maxsim_umma_pair: bad NM");
  }
}

int launch_score_umma_pair(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int nm, int m_tile_base,
                           int n_groups_real, void* scores, int64_t ld, cudaStream_t s) {
  switch (kind_of_dtype(h->corpus.dtype)) {
    case 0: return launch_pair_kind<0>(h, up, tq, nm, m_tile_base, n_groups_real, scores, ld, s);
    case 1: return launch_pair_kind<1>(h, up, tq, nm, m_tile_base, n_groups_real, scores, ld, s);
    case 2: return launch_pair_kind<2>(h, up, tq, nm, m_tile_base, n_groups_real, scores, ld, s);
    default: return set_error(h, B200MS_ESTATE, "maxsim_umma_pair: corpus dtype has no tcgen05 scorer");
  }
}

}  // namespace bms
