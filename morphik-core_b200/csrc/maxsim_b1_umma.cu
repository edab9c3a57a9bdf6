// maxsim_b1_umma.cu -- the 1-bit (sign / Hamming) MaxSim scorer on tcgen05 tensor cores.
//
// Same contract as maxsim_b1_kernel (SQL public.max_sim, core/vector_store/multi_vector_store.py:287-311): output
// S[g,p] = sum_{t in group g} max_r (128 - popcount(d_r ^ q_t)), exact integers.  The POPC formulation is pinned at the
// integer pipe's 16 popc/clk/SM (profiles/r01); sm_100a has no native 1-bit MMA (ptxas emulates mma.sync.b1 with legacy
// IMMA), so this kernel rewrites the Hamming distance as an int8 dot product the 5th-gen tensor cores can run:
//     q' = +1 / -1 per query bit,  d' = 1 / 0 per document bit   =>   <q', d'> = n11 - n01
//     ham(q,d) = n10 + n01 = popc(q) - <q', d'>                   =>   128 - ham = (128 - popc(q)) + <q', d'>
// so  max_r (128 - ham) = c_t + max_r <q'_t, d'_r>  with the per-token constant c_t = 128 - popc(q_t) (0 for padding).
//
// HBM traffic stays 16 B per patch vector: rows are fetched as packed bits (one coalesced 2 KB request per 128-row tile)
// and four "expander" warps inflate them to {0,1} bytes directly in the 128-byte-swizzled K-major shared-memory layout
// tcgen05.mma reads (thread r owns row r: 16 B -> 128 B, 8 x st.shared.v4, bit spreading with one IMAD + one LOP3 per
// 4 elements).  From there on the pipeline is the int8 MaxSim kernel: 4 x tcgen05.mma kind::i8 (128x128x32) per tile and
// query tile into one of 4 TMEM accumulators, per-thread running max in the epilogue, warp-shuffle sum at page ends.
// One 128-token query tile costs the same as one token, so 4 queries of 32 tokens ride for free.
// Bound: tensor pipe / expansion ALU, ~0.5 patch rows per clock per SM (vs 0.18 for the POPC kernel at one query).
#include "common.cuh"
#include "ptx.cuh"
#include "umma_tile.cuh"

namespace bms {

constexpr int kBThreads = 384;

// ------------------------------------------------------------------ query side: bits -> +-1 int8 rows + token constants
__global__ void __launch_bounds__(256)
b1_query_expand_kernel(const uint8_t* __restrict__ q_bits /*[rows,16]*/, const int32_t* __restrict__ group_ntok, int n_rows,
                       int8_t* __restrict__ out /*[rows,128]*/, int32_t* __restrict__ tok_const /*[rows]*/) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (row, byte of bits)
  const int row = idx >> 4, b = idx & 15;
  if (row >= n_rows) return;
  const bool real = (row & 31) < __ldg(group_ntok + (row >> 5));
  const uint32_t bits = q_bits[row * 16 + b];
  uint32_t lo = 0, hi = 0;  // elements 8b..8b+3 and 8b+4..8b+7 as int8 (MSB of the byte = first element)
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    lo |= (real ? (((bits >> (7 - e)) & 1u) ? 0x01u : 0xffu) : 0u) << (8 * e);
    hi |= (real ? (((bits >> (3 - e)) & 1u) ? 0x01u : 0xffu) : 0u) << (8 * e);
  }
  reinterpret_cast<uint2*>(out)[row * 16 + b] = make_uint2(lo, hi);
  if (b == 0) {
    const uint4 w = *reinterpret_cast<const uint4*>(q_bits + row * 16);
    tok_const[row] = real ? 128 - (__popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w)) : 0;
  }
}

template <int NM>
__global__ void __launch_bounds__(kBThreads, 1)
maxsim_b1_umma_kernel(const uint4* __restrict__ rows, int64_t n_rows, const __grid_constant__ CUtensorMap tmap_q,
                      const int32_t* __restrict__ tok_const, const int32_t* __restrict__ chunk_page,
                      const int32_t* __restrict__ unit_start, const int32_t* __restrict__ unit_end, int n_units,
                      int m_tile_base, int n_groups_real, int32_t* __restrict__ group_scores, int64_t ld, int num_stages) {
  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, NM * kSubtileBytes, kSubtileBytes, num_stages);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // full: one arrive per expander warp
  const uint32_t tmem_base = tile_prologue<false>(sm, warp, &tmap_q, nullptr, num_stages, 4, kNumAccum, 4);

  if (warp == 0) {
    // ================================================================ query tiles via TMA (+-1 int8, SWIZZLE_128B)
    if (lane == 0) {
      const uint64_t pol_q = policy_evict_last();
      mbar_expect_tx(sm.qfull, NM * kSubtileBytes);
#pragma unroll
      for (int m = 0; m < NM; ++m) tma_load_2d(&tmap_q, sm.qfull, sm.q + m * kSubtileBytes, 0, (m_tile_base + m) * kTileM, pol_q);
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (kind::i8, 4 K-steps of 32 per tile)
    constexpr uint32_t idesc = umma_idesc(1, kTileM, kTileN);
    constexpr uint32_t kTileDesc = kSubtileBytes >> 4;
    mbar_wait(sm.qfull, 0);
    tc_fence_after();
    const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.q));
    const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(sm.st));
    int stage = 0;
    uint32_t phase = 0, seq = 0;
    UnitWalk it;
    for (it.init(blockIdx.x, gridDim.x, unit_start, unit_end, n_units); it.valid(n_units);
         it.next(unit_start, unit_end, n_units)) {
      mbar_wait(&sm.full[stage], phase);
      tc_fence_after();
      const uint64_t bd = b_desc0 + uint64_t(uint32_t(stage) * kTileDesc);
#pragma unroll 1
      for (int m = 0; m < NM; ++m, ++seq) {
        const uint32_t buf = seq & (kNumAccum - 1);
        mbar_wait(&sm.tempty[buf], ((seq >> 2) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          umma_tile<1>(tmem_base + buf * kTileN, a_desc0 + uint64_t(uint32_t(m) * kTileDesc), bd, idesc);
          umma_commit(&sm.tfull[buf]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&sm.empty[stage]);
      __syncwarp();
      if (++stage == num_stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp >= 8) {
    // ================================================================ expanders: packed bits -> {0,1} int8, swizzled K-major
    const int r = (warp - 8) * 32 + lane;  // row of the tile this thread owns
    const uint32_t row_off = uint32_t(r >> 3) * 1024u + uint32_t(r & 7) * 128u;
    const uint32_t sw = uint32_t(r & 7);
    UnitWalk cur;
    cur.init(blockIdx.x, gridDim.x, unit_start, unit_end, n_units);
    UnitWalk pf = cur;
    constexpr int kRing = 8;
    uint4 ring[kRing];  // loads of the next 8 tiles stay in flight while the current one is expanded (DRAM latency >> tile time)
#pragma unroll
    for (int i = 0; i < kRing; ++i) {
      ring[i] = make_uint4(0, 0, 0, 0);
      if (pf.valid(n_units)) {
        const int64_t row = int64_t(pf.chunk()) * kGroup + r;
        if (row < n_rows) ring[i] = __ldg(rows + row);
        pf.next(unit_start, unit_end, n_units);
      }
    }
    int stage = 0;
    uint32_t phase = 0;
    while (cur.valid(n_units)) {
#pragma unroll
      for (int i = 0; i < kRing; ++i) {
        if (!cur.valid(n_units)) break;
        const uint4 mine = ring[i];
        ring[i] = make_uint4(0, 0, 0, 0);
        if (pf.valid(n_units)) {
          const int64_t row = int64_t(pf.chunk()) * kGroup + r;
          if (row < n_rows) ring[i] = __ldg(rows + row);
          pf.next(unit_start, unit_end, n_units);
        }
        mbar_wait(&sm.empty[stage], phase ^ 1);
        const uint32_t tile = smem_u32(sm.st) + uint32_t(stage) * kSubtileBytes + row_off;  // 32-bit shared address: st.shared, not generic ST
        const uint32_t words[4] = {mine.x, mine.y, mine.z, mine.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          // __brev: bit e%8 of (reversed) byte 3-b now holds element 8b + e%8 of this word's 32 elements
          const uint32_t rev = __brev(words[w]);
#pragma unroll
          for (int h = 0; h < 2; ++h) {  // 16-byte chunk c = 2w + h  <-  source bytes b = 2h, 2h+1 of the word
            // nibble n (bit e = element e) * 0x204081 puts bit k at k, k+7, k+14, k+21; masked with 0x01010101 that is one
            // element per byte.  (Only valid for 4-bit inputs: with 8 bits the shifted copies overlap and carry.)
            const uint32_t b0 = (rev >> (8 * (3 - 2 * h))) & 0xffu, b1 = (rev >> (8 * (2 - 2 * h))) & 0xffu;
            uint4 o;
            o.x = ((b0 & 0xfu) * 0x00204081u) & 0x01010101u;
            o.y = ((b0 >> 4) * 0x00204081u) & 0x01010101u;
            o.z = ((b1 & 0xfu) * 0x00204081u) & 0x01010101u;
            o.w = ((b1 >> 4) * 0x00204081u) & 0x01010101u;
            const uint32_t c = uint32_t(2 * w + h);
            st_shared_v4(tile + ((c ^ sw) << 4), o);
          }
        }
        fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.full[stage]);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
        cur.next(unit_start, unit_end, n_units);
      }
    }
  } else if (warp >= 4) {
    // ================================================================ epilogue (one warpgroup owns every query tile)
    const int quad = warp & 3;
    const uint32_t lane_base = tmem_base + (uint32_t(quad * 32) << 16);
    // one closed (group, page) run: the per-token constant, the 32-token sum, one store by lane 0
    const auto store = [&](int group, int cn, int page, int rm) {
      const int s = warp_sum(rm + cn);
      if (lane == 0) group_scores[int64_t(group) * ld + page] = s;
    };
    PageRun<int> runs[NM];
    int cnst[NM];
#pragma unroll
    for (int m = 0; m < NM; ++m) {
      const int group = (m_tile_base + m) * 4 + quad;
      cnst[m] = group < n_groups_real ? __ldg(tok_const + int64_t(m_tile_base + m) * kTileM + quad * 32 + lane) : 0;
    }
    const auto flush_all = [&]() {
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        const int group = (m_tile_base + m) * 4 + quad;
        runs[m].flush([&](int page, int rm) { store(group, cnst[m], page, rm); });
      }
    };
    uint32_t tile_seq = 0;
    int last_u = -1;
    UnitWalk it;
    for (it.init(blockIdx.x, gridDim.x, unit_start, unit_end, n_units); it.valid(n_units);
         it.next(unit_start, unit_end, n_units), ++tile_seq) {
      if (it.u != last_u) {  // new unit: units end on page boundaries
        flush_all();
        last_u = it.u;
      }
      int pg[4];
      tile_pages(chunk_page, it.chunk(), it.c1, pg);
#pragma unroll 1
      for (int m = 0; m < NM; ++m) {
        const uint32_t seq = tile_seq * NM + m;
        const uint32_t buf = seq & (kNumAccum - 1);
        const int group = (m_tile_base + m) * 4 + quad;
        PageRun<int> run;
        run.rm = 0;
        int cn = 0;
#pragma unroll
        for (int j = 0; j < NM; ++j)
          if (j == m) {
            run = runs[j];
            cn = cnst[j];
          }
        const auto release = [&] { mbar_arrive(&sm.tempty[buf]); };
        mbar_wait(&sm.tfull[buf], (seq >> 2) & 1);
        tc_fence_after();
        if (group < n_groups_real) {
          int cm[4];
          drain_accum(lane_base + buf * kTileN, cm, release);
          run.fold(pg, cm, [&](int page, int rm) { store(group, cn, page, rm); });
        } else {
          release_accum(release);
        }
#pragma unroll
        for (int j = 0; j < NM; ++j)
          if (j == m) runs[j] = run;
      }
    }
    flush_all();
  }
  tile_teardown<false>(warp, tmem_base);
}

template <int NM>
static int launch_b1_umma_one(b200ms_t* h, const CUtensorMap& tq, const int32_t* tok_const, int m_tile_base,
                              int n_groups_real, void* scores, int64_t ld, cudaStream_t s) {
  const Corpus& c = h->corpus;
  const int32_t* us = static_cast<const int32_t*>(h->unit_start.p);
  return launch_persistent(h, maxsim_b1_umma_kernel<NM>, "maxsim_b1_umma", kBThreads, NM * kSubtileBytes, kSubtileBytes, 8,
                           c.n_units, s, static_cast<const uint4*>(c.rows), c.n_rows, tq, tok_const,
                           static_cast<const int32_t*>(h->chunk_page.p), us, us + 1, c.n_units, m_tile_base, n_groups_real,
                           static_cast<int32_t*>(scores), ld);
}

int launch_score_b1_umma(b200ms_t* h, const void* q_bits, const int32_t* group_ntok_dev, int n_groups_real,
                         void* group_scores, int64_t ld, cudaStream_t s) {
  const int n_groups_padded = (n_groups_real + 3) & ~3;
  const int n_rows = n_groups_padded * kGroup;
  if (int e = reserve(h, h->b1_q_i8, size_t(n_rows) * 128 + 1024)) return e;
  if (int e = reserve(h, h->b1_tok_const, size_t(n_rows) * 4)) return e;
  int8_t* q_i8 = reinterpret_cast<int8_t*>((reinterpret_cast<uintptr_t>(h->b1_q_i8.p) + 1023) & ~uintptr_t(1023));
  int32_t* tok_const = static_cast<int32_t*>(h->b1_tok_const.p);
  b1_query_expand_kernel<<<(n_rows * 16 + 255) / 256, 256, 0, s>>>(static_cast<const uint8_t*>(q_bits), group_ntok_dev, n_rows,
                                                                  q_i8, tok_const);
  h->launches++;
  if (int e = check_cuda(h, cudaGetLastError(), "launch b1_query_expand")) return e;
  const int n_mtiles = n_groups_padded / 4;
  const CUtensorMap* tq;
  if (int e = query_tmap(h, q_i8, B200MS_I8, n_rows, kTileM, &tq)) return e;
  for (int base = 0; base < n_mtiles;) {
    const int rem = n_mtiles - base;
    int nm = 1;
    while (nm < rem && nm < 4) nm <<= 1;
    int e;
    switch (nm) {
      case 1: e = launch_b1_umma_one<1>(h, *tq, tok_const, base, n_groups_real, group_scores, ld, s); break;
      case 2: e = launch_b1_umma_one<2>(h, *tq, tok_const, base, n_groups_real, group_scores, ld, s); break;
      default: e = launch_b1_umma_one<4>(h, *tq, tok_const, base, n_groups_real, group_scores, ld, s); break;
    }
    if (e) return e;
    base += nm;
  }
  return B200MS_OK;
}

}  // namespace bms
