// maxsim_rowm.cu -- the lone-query MaxSim scan with the ROLES OF THE MMA OPERANDS SWAPPED: patch rows are M, query tokens are N.
//
// Same contract as maxsim_umma_kernel<KIND,1> (float / int8 / fp8 MaxSim, colpali_engine score_multi_vector called at
// core/vector_store/fast_multivector_store.py:553-555) and maxsim_b1_umma_kernel (SQL public.max_sim,
// core/vector_store/multi_vector_store.py:287-311) for a scan that carries at most 64 query tokens -- the single-query
// regime of BASELINE configs[0] / configs[2], where the scan is supposed to be HBM-bound.
//
// Why a second orientation.  With the query as the M operand (maxsim_umma.cu) a lone 32-token query fills 32 of the 128
// accumulator lanes, the tensor core still pays for 128 x 128, and -- TMEM lanes being private to one warp of a warpgroup --
// ONE epilogue warp walks all 128 columns of every tile: a serial load -> max chain of ~700 cycles per tile.  That hides
// behind a 32 KB bf16 tile (0.98 of HBM) but not behind a 16 KB int8 / fp8 tile (0.68-0.87 of HBM, profiles/r02) and not at
// all behind a 2 KB tile of sign bits (0.10).  Here a tile is  D[128 patch rows, 32*NG tokens] = A[rows] * B[tokens]^T :
//   * tcgen05.mma 128 x 32 x 32B costs 16 cycles per K step instead of 64 (B300_MICROARCH.md "tcgen05 floor"),
//   * lane quadrant w of the accumulator = chunk w of the tile (32 consecutive patch rows), so the FOUR epilogue warps each
//     read 32 lanes x 32 columns (one tcgen05.ld) and fold it into a per-thread running max over (row slot, token):
//     32 max instructions per warp and tile, all four warps in parallel,
//   * the max over the ROWS of a page is a max over lanes and over warps, taken once per page instead of once per tile: a
//     31-shuffle butterfly leaves token t's maximum over the warp's rows in lane t, the four warps meet in a small shared-memory
//     table (atomicMax per token + a chunk counter per page; the warp that completes the page's chunk count sums the tokens
//     and writes the score).  Pages are whole inside a CTA's unit, so no global atomics are needed.
//
// KIND 0 bf16, 1 int8, 2 fp8 e4m3: patch tiles arrive by TMA exactly as in maxsim_umma.cu (up to 14 stages: 16 KB tiles need
//   > 128 KB in flight per SM), A and B from shared memory.
// KIND 3 sign bits: rows stay 16 B in HBM.  A bulk-copy ring brings raw bits into shared memory (16 KB slots = 8 tiles, one
//   request per contiguous run); eight expander warps -- two per TMEM lane quadrant, alternating tiles, one thread per patch row --
//   turn 16 B of bits into 32 words of int8 (ONE AND per word: bit m+8i stays in place as 2^m, the +-1 query carries the
//   inverse weight 2^(6-m), every product is +-64; the K order inside a 32-bit word is permuted, element 4m+i <- bit m+8i,
//   and the query is expanded with the same permutation, which a dot product cannot see) and store
//   them with ONE tcgen05.st straight into TMEM, where tcgen05.mma kind::i8 reads its A operand (no shared-memory store, no
//   swizzle, no proxy fence).  128 - ham = (128 - popc(q)) + <q', d'> as in maxsim_b1_umma.cu.
// Two epilogue warps per lane quadrant alternate tiles as well: every per-tile loop in this kernel is a serial chain inside a
//   lone warp that pays full latency per instruction (ncu: ~10 cycles each), so the loops are kept short -- the MMA issuer and
//   the expanders only count tiles, the epilogue does its page bookkeeping once per 8-tile block from two ballots (chunk ->
//   page ids prefetched one block ahead; page extents come from the masks, not from page_start) and has a fast path for blocks
//   that lie inside one page.
// Results: bit-identical to the query-as-M kernels (integer kinds exact; float kinds take the same max and the same
// lane-order warp sum).  Measured (65536 pages x 1024, one 32-token query, B200): bf16 2.37 ms = 7.25 TB/s (query-as-M: 2.50),
// int8 / fp8 1.17-1.27 ms = 6.8-7.4 TB/s (1.47), sign bits 0.97 ms (POPC kernel 1.57); profiles/r02/README.md section 8.
#include <climits>

#include "common.cuh"
#include "ptx.cuh"
#include "umma_tile.cuh"

namespace bms {

constexpr int kRmSlots = 128;         // page slots of the cross-warp combine table: a warp is at most ~2 blocks = 64 pages away from
                                      // the slowest one (8 accumulators = 8 tiles ahead; a finished page is flushed at the next block)
constexpr int kRmRawGroups = 6;       // KIND 3: raw-bit ring, slots of 8 tiles = 16 KB, one bulk copy per contiguous run (a 2 KB copy
constexpr int kRmGroupTiles = 8;      //   per tile left the expanders waiting for data although 48 were in flight; measured +4 %)
constexpr uint32_t kRmRawTile = 128 * 16;
constexpr uint32_t kRmRawGroupBytes = kRmGroupTiles * kRmRawTile;
constexpr int kRmMaxStages = 14;      // TMA kinds: 16 / 32 KB patch tiles in flight (HBM latency x bandwidth wants > 128 KB per SM)
constexpr int kRmARing = 8;           // KIND 3: expanded A tiles in TMEM (32 columns each, columns [256, 512))
constexpr uint32_t kRmAColBase = 256;

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {  // no arrival: more bytes for the current phase
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// mbarrier wait with a suspend-time hint: the thread sleeps inside the try_wait until the phase completes (or ~2 us pass) instead of
// coming back every ~90 cycles.  In this kernel the pollers share their SM sub-partition's issue slots with the warps that
// work (ncu: ~1050 warp instructions per 128-row tile, 18 % of them polling); A/B against plain polling: neutral to +1 %
// (profiles/r02/rowm_hint_ab.jsonl, measured with a runtime switch that is gone again).
__device__ __forceinline__ void rm_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(2000u)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
// registers -> TMEM: this warp's 32 lanes x 32 consecutive 32-bit columns.  Whole warp; tmem_st_wait() before signalling.
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]^T, kind::i8: A = 128 lanes (rows) x 8 columns (32 B of K) at a_tmem
__device__ __forceinline__ void umma_ts_i8(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// shared-memory atomics by 32-bit shared address (a pointer carved out of the dynamic shared array compiles to GENERIC atomics)
__device__ __forceinline__ void smem_red_max(uint32_t addr, int v) {
  asm volatile("red.shared.max.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ int smem_atom_add(uint32_t addr, int v) {
  int old;
  asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ int smem_atom_exch(uint32_t addr, int v) {
  int old;
  asm volatile("atom.shared.exch.b32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void fence_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }
__device__ __forceinline__ float acc_lowest(float) { return -__int_as_float(0x7f800000); }  // -inf
__device__ __forceinline__ int acc_lowest(int) { return INT_MIN; }

// order-preserving int key of an accumulator value (atomicMax in shared memory works on ints)
__device__ __forceinline__ int rm_key(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ int rm_key(int v) { return v; }
__device__ __forceinline__ float rm_val(int k, float) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }
__device__ __forceinline__ int rm_val(int k, int) { return k; }

// r[i] of lane l = value of (row slot l, token i).  Returns, in lane t, the maximum over all 32 lanes of token t.
template <int N, typename Acc>
__device__ __forceinline__ void rm_fold(Acc (&r)[32], int lane) {
  constexpr int H = N / 2;
  const bool upper = (lane & H) != 0;
#pragma unroll
  for (int i = 0; i < H; ++i) {
    const Acc send = upper ? r[i] : r[i + H];
    const Acc keep = upper ? r[i + H] : r[i];
    r[i] = acc_max(keep, __shfl_xor_sync(0xffffffffu, send, H));
  }
}
template <typename Acc>
__device__ __forceinline__ Acc rm_lane_transpose_max(Acc (&r)[32], int lane) {
  rm_fold<32>(r, lane);
  rm_fold<16>(r, lane);
  rm_fold<8>(r, lane);
  rm_fold<4>(r, lane);
  rm_fold<2>(r, lane);
  return r[0];
}

// the CTA's tile sequence: units blockIdx.x, +gridDim.x, ...; 128-row tiles inside a unit (every warp role walks it).
// The chunk range of the NEXT unit is loaded one unit ahead, so its DRAM latency hides behind the current unit's tiles.
struct RmTiles {
  int u, t, n_tiles, c0, c1;
  int nc0, nc1;
  __device__ __forceinline__ void fetch_next(const int32_t* us, const int32_t* ue, int n_units) {
    const int nu = u + int(gridDim.x);
    nc0 = nc1 = 0;
    if (nu < n_units) {
      nc0 = __ldg(us + nu);
      nc1 = __ldg(ue + nu);
    }
  }
  __device__ __forceinline__ void advance(const int32_t* us, const int32_t* ue, int n_units) {
    u += int(gridDim.x);
    c0 = nc0;
    c1 = nc1;
    n_tiles = (c1 - c0 + 3) >> 2;
    t = 0;
    fetch_next(us, ue, n_units);
  }
  __device__ __forceinline__ void start(const int32_t* us, const int32_t* ue, int n_units) {
    u = int(blockIdx.x);
    c0 = c1 = 0;
    if (u < n_units) {
      c0 = __ldg(us + u);
      c1 = __ldg(ue + u);
    }
    n_tiles = (c1 - c0 + 3) >> 2;
    t = 0;
    fetch_next(us, ue, n_units);
    while (u < n_units && n_tiles == 0) advance(us, ue, n_units);
  }
  __device__ __forceinline__ bool valid(int n_units) const { return u < n_units; }
  __device__ __forceinline__ void next(const int32_t* us, const int32_t* ue, int n_units) {
    if (++t == n_tiles) {
      advance(us, ue, n_units);
      while (u < n_units && n_tiles == 0) advance(us, ue, n_units);
    }
  }
  __device__ __forceinline__ int chunk0() const { return c0 + 4 * t; }
};

// chunk -> page lookahead of an epilogue warp: lane l holds chunk_page[base + l] for a block of 32 chunks (8 tiles); the next
// block (of this unit, or the first of the next unit) is loaded while the current one is consumed.  A per-tile __ldg here was
// THE limiter of the 16 KB-tile scans: chunk_page streams from DRAM, a sector miss every other tile put ~1 us of latency into
// a chain every tile of the warp has to pass (415 ns per tile measured, whatever the tile held).
struct RmPages {
  int cur, nxt, nxt_base;
  __device__ __forceinline__ static int load(const int32_t* chunk_page, int base, int limit, int lane) {
    return base + lane < limit ? __ldg(chunk_page + base + lane) : -1;
  }
  // Two steps on purpose.  take(): cur <- the block loaded one block ago (a synchronous reload only if the lookahead guessed
  // wrong).  prefetch(): issue the next block's load AFTER every use of cur in the block setup -- ptxas shares scoreboards, and
  // with the load issued first the first consumer of cur waited for the NEW load as well (a DRAM round trip per block, ncu).
  __device__ __forceinline__ void take(const RmTiles& it, const int32_t* chunk_page, int lane) {
    const int base = it.c0 + 4 * it.t;  // it.t % 8 == 0
    if (nxt_base != base) {
      nxt = load(chunk_page, base, it.c1, lane);
      nxt_base = base;
    }
    cur = nxt;
  }
  __device__ __forceinline__ void prefetch(const RmTiles& it, const int32_t* chunk_page, int n_units, int lane) {
    const int base = it.c0 + 4 * it.t;
    if (it.t + 8 < it.n_tiles) {
      nxt_base = base + 32;
      nxt = load(chunk_page, nxt_base, it.c1, lane);
    } else if (it.u + int(gridDim.x) < n_units) {
      nxt_base = it.nc0;
      nxt = load(chunk_page, nxt_base, it.nc1, lane);
    } else {
      nxt_base = -1;
    }
  }
  __device__ __forceinline__ int page_of(const RmTiles& it, int j) const {
    return __shfl_sync(0xffffffffu, cur, 4 * (it.t & 7) + j);
  }
};

// ------------------------------------------------------------------ KIND 3 query side: bits -> +-1 int8 rows (permuted K) + token constants
__global__ void __launch_bounds__(256)
rowm_query_expand_kernel(const uint32_t* __restrict__ q_words /*[rows,4]*/, const int32_t* __restrict__ group_ntok, int n_rows,
                         uint4* __restrict__ out /*[rows,128 B]*/, int32_t* __restrict__ tok_const /*[rows]*/) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (row, 32-bit word)
  const int row = idx >> 2, w = idx & 3;
  if (row >= n_rows) return;
  const bool real = (row & 31) < __ldg(group_ntok + (row >> 5));
  const uint32_t x = __ldg(q_words + idx);
  // The row expanders leave bit m+8i of a word IN PLACE (byte i of output word m = 2^m * bit for m <= 6, one AND per word;
  // bit 7 is the int8 sign, so m = 7 is shifted down to 2^6): the query carries the inverse weight W_m = 2^(6-m) (W_7 = 1), every
  // product is +-64 and the accumulator is 64 * (n11 - n01), exactly.
  uint32_t o[8];
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const uint32_t t = (x >> m) & 0x01010101u;                     // element 4m+i <- bit m+8i  (same as the row expanders)
    const uint32_t w = m < 7 ? (1u << (6 - m)) : 1u;
    const uint32_t pos = t * w, neg = (t ^ 0x01010101u) * ((256u - w) & 0xffu);  // bit 1 -> +W, bit 0 -> -W (two's complement byte)
    o[m] = real ? (pos | neg) : 0u;                                // padding token -> 0
  }
  out[idx * 2] = make_uint4(o[0], o[1], o[2], o[3]);
  out[idx * 2 + 1] = make_uint4(o[4], o[5], o[6], o[7]);
  if (w == 0) {
    const uint4 q = *reinterpret_cast<const uint4*>(q_words + idx);
    tok_const[row] = real ? 128 - (__popc(q.x) + __popc(q.y) + __popc(q.z) + __popc(q.w)) : 0;
  }
}

template <int KIND>
struct RmTraits {
  static constexpr int kMmaKind = KIND == 3 ? 1 : KIND;
  using K = Kind<kMmaKind>;
  using Acc = typename K::Acc;
  // warps 0-3: producer / MMA issuer / TMEM allocator / idle; 4-11: two epilogue sets (set e takes the tiles with seq % 2 == e);
  // KIND 3: 12-19 expanders
  static constexpr int kThreads = KIND == 3 ? 640 : 384;
};

template <int KIND, int NG>
__global__ void __launch_bounds__(RmTraits<KIND>::kThreads, 1)
maxsim_rowm_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
                   const uint8_t* __restrict__ raw_rows, int64_t n_rows, const int32_t* __restrict__ tok_const,
                   const int32_t* __restrict__ chunk_page, const int32_t* __restrict__ unit_start,
                   const int32_t* __restrict__ unit_end, int n_units, int n_groups_real, const uint32_t* __restrict__ clamp_bits,
                   typename RmTraits<KIND>::Acc* __restrict__ group_scores, int64_t ld, int num_stages) {
  using T = RmTraits<KIND>;
  using K = typename T::K;
  using Acc = typename T::Acc;
  constexpr int kKSteps = K::kKSteps;
  constexpr uint32_t kQPanel = NG * 4096;  // one K panel of the query operand: 32*NG rows x 128 B
  constexpr uint32_t kQBytes = K::kPanels * kQPanel;
  constexpr uint32_t kAccCols = 32 * NG;
  constexpr int kAcc = (KIND == 3 && NG == 2) ? 4 : 8;  // TMEM accumulators (KIND 3 keeps columns [256,512) for the A ring)

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_q = smem;
  uint8_t* smem_st = smem + ((kQBytes + 1023) & ~1023u);  // TMA kinds: num_stages patch tiles; KIND 3: the raw-bit ring
  uint8_t* smem_rawring = smem_st;
  int* pm = reinterpret_cast<int*>(smem_st + (KIND == 3 ? size_t(kRmRawGroups) * kRmRawGroupBytes : size_t(num_stages) * K::kTileBytes));
  int* cnt = pm + NG * kRmSlots * 32;  // pm: [NG][kRmSlots][32] per-token maxima; cnt: [kRmSlots] chunks merged so far
  uint64_t* bars = reinterpret_cast<uint64_t*>(cnt + kRmSlots);  // kBarrierBytes: the arrays below + TMEM slot + tile count
  uint64_t* full = bars;            // [num_stages] A tile ready for the MMA  (TMA bytes | KIND 3: 4 expander warps)
  uint64_t* empty = bars + 16;      // [num_stages] MMA done with the stage
  uint64_t* tfull = bars + 32;      // [kAcc]       MMA -> epilogue
  uint64_t* tempty = bars + 40;     // [kAcc]       epilogue -> MMA (4 warps)
  uint64_t* qfull = bars + 48;
  uint64_t* rfull = bars + 56;      // [kRmRawGroups] KIND 3: raw bits of a group of 8 tiles landed
  uint64_t* rempty = bars + 120;    // [kRmRawGroups] KIND 3: the expander warps have read all of the group
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 184);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    if (KIND != 3) prefetch_tmap(&tmap_rows);
    prefetch_tmap(&tmap_q);
    for (int i = 0; i < num_stages; ++i) {
      mbar_init(&full[i], KIND == 3 ? 4 : 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < kAcc; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    mbar_init(qfull, 1);
    if (KIND == 3)
      for (int i = 0; i < kRmRawGroups; ++i) {
        mbar_init(&rfull[i], 1);                    // the producer's arrive once the whole group is requested (+ its bytes)
        mbar_init(&rempty[i], 4 * kRmGroupTiles);   // every expander warp, once per tile it reads
      }
    fence_mbar_init();
  }
  for (int i = threadIdx.x; i < NG * kRmSlots * 32 + kRmSlots; i += blockDim.x) pm[i] = i < NG * kRmSlots * 32 ? INT_MIN : 0;
  // tiles this CTA will stream: the MMA issuer and the expanders only need the COUNT (their per-tile loops must stay a few
  // dozen instructions: a lone warp pays full latency for every instruction, ncu showed 8-10 cycles each)
  int* total_slot = reinterpret_cast<int*>(tmem_slot + 1);
  if (threadIdx.x == 0) *total_slot = 0;
  __syncthreads();
  {
    int mine = 0;
    for (int u = int(blockIdx.x) + int(threadIdx.x) * int(gridDim.x); u < n_units; u += int(blockDim.x) * int(gridDim.x))
      mine += (__ldg(unit_end + u) - __ldg(unit_start + u) + 3) >> 2;
    if (mine) atomicAdd(total_slot, mine);
  }
  if (warp == 2) tmem_alloc_512(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t total_tiles = uint32_t(*total_slot);

  if (warp == 0) {
    // ================================================================ producer: query tile once, then the patch tiles
    if (lane == 0) {
      const uint64_t pol_rows = policy_evict_first();
      const uint64_t pol_q = policy_evict_last();
      mbar_expect_tx(qfull, kQBytes);
#pragma unroll
      for (int p = 0; p < K::kPanels; ++p) tma_load_2d(&tmap_q, qfull, smem_q + p * kQPanel, p * K::kPanelElems, 0, pol_q);
      RmTiles it;
      it.start(unit_start, unit_end, n_units);
      if constexpr (KIND == 3) {
        // groups of 8 consecutive tiles of the CTA's sequence share a 16 KB slot; tiles that are contiguous in HBM (same unit)
        // travel as ONE bulk copy, a group that crosses a unit boundary as two
        int rg = 0, in_group = 0, run_first = 0, run_tiles = 0;
        uint32_t gphase = 0;
        int64_t run_row0 = 0;
        auto issue_run = [&]() {
          if (run_tiles == 0) return;
          const int64_t left = (n_rows - run_row0) * 16;
          const int64_t want = int64_t(run_tiles) * kRmRawTile;
          const uint32_t bytes = uint32_t(left < want ? left : want);
          mbar_expect_tx_only(&rfull[rg], bytes);
          bulk_load_1d(smem_rawring + rg * kRmRawGroupBytes + run_first * kRmRawTile, raw_rows + run_row0 * 16, bytes, &rfull[rg],
                       pol_rows);
          run_tiles = 0;
        };
        for (; it.valid(n_units); it.next(unit_start, unit_end, n_units)) {
          const int64_t row0 = int64_t(it.chunk0()) * kGroup;
          if (in_group == 0) rm_wait(&rempty[rg], gphase ^ 1);
          if (run_tiles > 0 && row0 == run_row0 + int64_t(run_tiles) * 128) {
            ++run_tiles;
          } else {
            issue_run();
            run_first = in_group;
            run_row0 = row0;
            run_tiles = 1;
          }
          if (++in_group == kRmGroupTiles) {
            issue_run();
            mbar_arrive(&rfull[rg]);
            in_group = 0;
            if (++rg == kRmRawGroups) {
              rg = 0;
              gphase ^= 1;
            }
          }
        }
        if (in_group > 0) {
          issue_run();
          mbar_arrive(&rfull[rg]);
        }
      } else {
        int stage = 0;
        uint32_t phase = 0;
        for (; it.valid(n_units); it.next(unit_start, unit_end, n_units)) {
          rm_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], K::kTileBytes);
          uint8_t* dst = smem_st + size_t(stage) * K::kTileBytes;
          const int row0 = it.chunk0() * kGroup;
#pragma unroll
          for (int p = 0; p < K::kPanels; ++p)
            tma_load_2d(&tmap_rows, &full[stage], dst + p * kSubtileBytes, p * K::kPanelElems, row0, pol_rows);
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer: D[128 rows, 32*NG tokens] per tile
    constexpr uint32_t idesc = umma_idesc(T::kMmaKind, kTileN, int(kAccCols));
    constexpr uint32_t kTileDesc = K::kTileBytes >> 4;
    if (elect_one()) {  // one thread runs the whole loop: no per-tile elect / warp sync
      rm_wait(qfull, 0);
      tc_fence_after();
      const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(smem_st));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(smem_q));
      uint32_t stage = 0, phase = 0;
      for (uint32_t seq = 0; seq < total_tiles; ++seq) {
        const uint32_t buf = seq & (kAcc - 1);
        rm_wait(&full[stage], phase);
        rm_wait(&tempty[buf], ((seq / kAcc) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * kAccCols;
#pragma unroll
        for (int ks = 0; ks < kKSteps; ++ks) {  // 32 B of K per step; 4 steps per 128 B panel
          const uint32_t off_b = ((ks >> 2) * kQPanel + (ks & 3) * 32) >> 4;
          if constexpr (KIND == 3) {  // A = the expanded tile in TMEM: 8 columns (32 B of K) per step
            umma_ts_i8(d_tmem, tmem_base + kRmAColBase + stage * 32u + uint32_t(ks) * 8u, b_desc0 + off_b, idesc, ks != 0);
          } else {
            const uint64_t ad = a_desc0 + uint64_t(stage * kTileDesc);
            const uint32_t off_a = ((ks >> 2) * kSubtileBytes + (ks & 3) * 32) >> 4;
            umma_ss<T::kMmaKind>(d_tmem, ad + off_a, b_desc0 + off_b, idesc, ks != 0);
          }
        }
        umma_commit(&tfull[buf]);
        umma_commit(&empty[stage]);
        if (++stage == uint32_t(num_stages)) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ================================================================ epilogue: warp `quad` owns chunk `quad` of every tile
    // Each epilogue warp is alone on its SM sub-partition and every tile passes through it, so the instructions of this loop
    // are a serial chain per tile: keep it short (ncu: 229 instructions per tile and warp = 950 cycles bounded every kind;
    // the page bookkeeping is done once per 8-tile block with a ballot, the running max has no select).
    const int quad = warp & 3;
    const uint32_t eset = uint32_t(warp - 4) >> 2;  // two warps per lane quadrant, alternate tiles: the chain below gets 2 tile times
    const uint32_t lane_base = tmem_base + (uint32_t(quad * 32) << 16);
    const uint32_t pm_s = smem_u32(pm) + uint32_t(lane) * 4u, cnt_s = smem_u32(cnt);
    Acc rm[NG][32];
    int cn[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) cn[g] = (KIND == 3 && g < n_groups_real) ? __ldg(tok_const + g * 32 + lane) : 0;
    int cp = -1, cord = 0, ccount = 0;  // page this warp is accumulating, its ordinal in the CTA's page sequence, chunks so far
    // Positions in the CTA's chunk sequence (every warp sees every block's masks, so all of this is register arithmetic -- a
    // page_start load per page put a DRAM round trip on the scoreboards the tile loop waits on):
    int g_base = 0, last_change_g = -1;  // index of this block's chunk 0; index of the last page change before this block
    int cp_start_g = 0, cp_end_g = -1;   // [first chunk, one past the last chunk) of page cp; end < 0: not seen yet
    int last_pg = -1, ord_base = 0;      // page of the last chunk of the previous block, page changes before this block
    uint32_t cmask = 0, vmask = 0;      // this block: chunk i starts a new page / chunk i exists
    uint32_t seq = 0;

    auto flush = [&]() {
      const uint32_t slot = uint32_t(cord) & (kRmSlots - 1);
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const Acc r = rm_lane_transpose_max(rm[g], lane);
        smem_red_max(pm_s + (uint32_t(g) * kRmSlots + slot) * 128u, rm_key(r));
      }
      fence_cta();
      __syncwarp();
      int old = 0;
      if (lane == 0) old = smem_atom_add(cnt_s + slot * 4u, ccount);
      old = __shfl_sync(0xffffffffu, old, 0);
      const int total = cp_end_g - cp_start_g;  // chunks of page cp
      if (old + ccount == total) {  // this warp brought the page's last chunks: every warp's maxima are in the table
        fence_cta();
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          const int k = smem_atom_exch(pm_s + (uint32_t(g) * kRmSlots + slot) * 128u, INT_MIN);
          if (g < n_groups_real) {
            Acc v = rm_val(k, Acc(0));
            if (KIND != 3) v = clamp_token_max(clamp_bits, cp, v);
            if constexpr (KIND == 3) v = v >> 6;  // accumulators are 64 * (n11 - n01): exact
            const Acc sum = warp_sum(Acc(v + Acc(cn[g])));
            if (lane == 0) group_scores[int64_t(g) * ld + cp] = sum;
          }
        }
        if (lane == 0) smem_atom_exch(cnt_s + slot * 4u, 0);
      }
    };

    auto adopt = [&](int pg, uint32_t i) {  // this warp's chunk i of the current block belongs to another page than cp
      if (cp >= 0) flush();
      const uint32_t upto = (2u << i) - 1u;  // bits 0..i (i = 31: wraps to all ones)
      const uint32_t le = cmask & upto, gt = cmask & ~upto;
      cp = pg;
      cord = ord_base + __popc(le);
      ccount = 0;
      cp_start_g = le ? g_base + 31 - __clz(le) : last_change_g;
      cp_end_g = gt ? g_base + __ffs(gt) - 1 : -1;
#pragma unroll
      for (int g = 0; g < NG; ++g)
#pragma unroll
        for (int c = 0; c < 32; ++c) rm[g][c] = acc_lowest(Acc(0));
    };

    RmTiles it;
    it.start(unit_start, unit_end, n_units);
    RmPages pages;
    pages.nxt_base = -1;
    pages.nxt = pages.cur = -1;
    for (; it.valid(n_units); it.next(unit_start, unit_end, n_units), ++seq) {
      const int tt = it.t & 7;
      if (tt == 0) {  // a block of <= 8 tiles = 32 chunks: lane l looks at chunk l
        ord_base += __popc(cmask);
        if (cmask) last_change_g = g_base + 31 - __clz(cmask);
        g_base += __popc(vmask);
        pages.take(it, chunk_page, lane);
        int prev = __shfl_up_sync(0xffffffffu, pages.cur, 1);
        if (lane == 0) prev = last_pg;
        const bool valid = pages.cur >= 0;
        vmask = __ballot_sync(0xffffffffu, valid);
        cmask = __ballot_sync(0xffffffffu, valid && pages.cur != prev);
        last_pg = __shfl_sync(0xffffffffu, pages.cur, __popc(vmask) - 1);  // valid chunks are a prefix of the block
        pages.prefetch(it, chunk_page, n_units, lane);
        if (cp >= 0 && cp_end_g < 0 && cmask != 0u) cp_end_g = g_base + __ffs(cmask) - 1;  // the first change ends page cp
        if (cp >= 0 && cp_end_g >= 0 && cp_end_g <= g_base) {
          // page cp ended before this block: hand its maxima over NOW.  Waiting for this warp's next chunk of another page can
          // take arbitrarily long when its lane quadrant has no rows for a while (runs of units that end in partial tiles), and
          // the page-slot table is only kRmSlots ordinals deep.
          flush();
          cp = -1;
        }
        if (vmask == 0xffffffffu && (cmask & ~1u) == 0u) {
          // fast path: 8 whole tiles of ONE page (it may begin at this block's first chunk -- 1024-row pages are exactly one
          // block): at most one adoption, then four owned tiles without bookkeeping
          if (last_pg != cp) adopt(last_pg, 0u);
          const uint32_t first = seq + ((seq ^ eset) & 1u);
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) {
            const uint32_t sq = first + 2u * k;
            const uint32_t buf = sq & (kAcc - 1);
            rm_wait(&tfull[buf], (sq / kAcc) & 1);
            tc_fence_after();
#pragma unroll
            for (int g = 0; g < NG; ++g) {
              uint32_t v[32];
              tmem_ld_32x32(lane_base + buf * kAccCols + g * 32, v);
              tmem_ld_wait();
              if (g == NG - 1) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[buf]);
              }
#pragma unroll
              for (int c = 0; c < 32; ++c) rm[g][c] = acc_max(rm[g][c], acc_from_bits(v[c], Acc(0)));
            }
          }
          ccount += 4;
          it.t += 7;
          seq += 7;
          continue;
        }
      }
      if ((seq & 1u) != eset) continue;
      const uint32_t i = uint32_t(4 * tt + quad);
      const bool mine = (vmask >> i) & 1u;
      const uint32_t buf = seq & (kAcc - 1);
      rm_wait(&tfull[buf], (seq / kAcc) & 1);
      tc_fence_after();
      if (mine) {
        const int my_pg = __shfl_sync(0xffffffffu, pages.cur, int(i));
        if (my_pg != cp) adopt(my_pg, i);
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          uint32_t v[32];
          tmem_ld_32x32(lane_base + buf * kAccCols + g * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 32; ++c) rm[g][c] = acc_max(rm[g][c], acc_from_bits(v[c], Acc(0)));
        }
        ++ccount;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
    if (cp >= 0) {
      if (cp_end_g < 0) cp_end_g = g_base + __popc(vmask);  // the page runs to the end of this CTA's stream
      flush();
    }
  } else if (KIND == 3 && warp >= 12) {
    // ================================================================ expanders: 2 KB of sign bits -> A tile in TMEM
    // Warp (quad, par): rows quad*32 .. +31 (its TMEM lane quadrant) of the tiles with seq % 2 == par; thread = one row:
    // 16 B of bits -> 32 words of {0,1} bytes (word 8w+m = (x_w >> m) & 0x01010101: element 4m+i <- bit m+8i) -> one
    // tcgen05.st of 32 columns.  No shared-memory store, no swizzle, no proxy fence: the tensor core reads A from TMEM.
    const int quad = warp & 3, par = (warp - 12) >> 2;
    const uint32_t raw0 = smem_u32(smem_rawring) + uint32_t(quad * 32 + lane) * 16u;
    const uint32_t a_lane = tmem_base + (uint32_t(quad * 32) << 16) + kRmAColBase;
    static_assert((kRmARing & (kRmARing - 1)) == 0 && kRmGroupTiles == 8, "ring sizes");
    uint32_t rs = 0, rphase = 0, prev_g = 0;
    for (uint32_t seq = uint32_t(par); seq < total_tiles; seq += 2) {
      const uint32_t g = seq >> 3;
      if (g != prev_g) {  // next group of 8 tiles: next raw slot
        prev_g = g;
        if (++rs == uint32_t(kRmRawGroups)) {
          rs = 0;
          rphase ^= 1u;
        }
      }
      const uint32_t stage = seq & uint32_t(kRmARing - 1), phase = (seq / uint32_t(kRmARing)) & 1u;
      rm_wait(&rfull[rs], rphase);
      const uint4 bits = ld_shared_v4(raw0 + rs * kRmRawGroupBytes + (seq & 7u) * kRmRawTile);
      __syncwarp();
      if (lane == 0) mbar_arrive(&rempty[rs]);
      uint32_t v[32];
      const uint32_t x[4] = {bits.x, bits.y, bits.z, bits.w};
#pragma unroll
      for (int w = 0; w < 4; ++w) {
#pragma unroll
        for (int m = 0; m < 7; ++m) v[8 * w + m] = x[w] & (0x01010101u << m);  // 2^m * bit, in place: one LOP3 per word
        v[8 * w + 7] = (x[w] >> 1) & 0x40404040u;                                // bit 7 would be the sign: park it at 2^6
      }
      rm_wait(&empty[stage], phase ^ 1);
      tc_fence_after();
      tmem_st_32x32(a_lane + stage * 32u, v);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[stage]);
    }
  }
  tile_teardown<false>(warp, tmem_base);
}

// Resident shared memory: the query panels (1 KB aligned), the [NG][kRmSlots][32] maxima table and the kRmSlots counters.
// KIND 0-2 stream patch tiles through up to kRmMaxStages stages; KIND 3 adds the raw-bit ring and its kRmARing stages are
// A tiles in TMEM.
template <int KIND, int NG>
static int launch_rowm_one(b200ms_t* h, const CUtensorMap& tq, const int32_t* tok_const, int n_groups_real,
                           const uint32_t* clamp_bits, void* scores, int64_t ld, cudaStream_t s) {
  using T = RmTraits<KIND>;
  using K = typename T::K;
  const Corpus& c = h->corpus;
  uint32_t resident = ((K::kPanels * NG * 4096u + 1023u) & ~1023u) + NG * kRmSlots * 32 * 4 + kRmSlots * 4;
  if (KIND == 3) resident += kRmRawGroups * kRmRawGroupBytes;
  const int32_t* us = static_cast<const int32_t*>(h->unit_start.p);
  return launch_persistent(h, maxsim_rowm_kernel<KIND, NG>, "maxsim_rowm", T::kThreads, resident,
                           KIND == 3 ? 0u : K::kTileBytes, KIND == 3 ? kRmARing : kRmMaxStages, c.n_units, s, c.tmap, tq,
                           static_cast<const uint8_t*>(c.rows), c.n_rows, tok_const,
                           static_cast<const int32_t*>(h->chunk_page.p), us, us + 1, c.n_units, n_groups_real, clamp_bits,
                           static_cast<typename T::Acc*>(scores), ld);
}

// Full scan of the attached corpus with n_groups_real <= kRowmMaxGroups 32-token query groups.  q_packed: the packed query
// rows in the corpus dtype (sign bits for B200MS_B1, with ntok_dev = real tokens per group).
int launch_score_rowm(b200ms_t* h, const void* q_packed, int n_groups_real, const int32_t* ntok_dev, const uint32_t* clamp_bits,
                      void* group_scores, int64_t ld, cudaStream_t s) {
  const Corpus& c = h->corpus;
  if (n_groups_real < 1 || n_groups_real > kRowmMaxGroups) return set_error(h, B200MS_EINVAL, "maxsim_rowm: 1 or 2 query groups");
  const int ng = n_groups_real;
  const int n_groups_padded = (n_groups_real + 3) & ~3;
  const int n_q_rows = n_groups_padded * kGroup;
  const void* q_rows = q_packed;
  int q_dtype = c.dtype;
  const int32_t* tok_const = nullptr;
  if (c.dtype == B200MS_B1) {
    if (!ntok_dev) return set_error(h, B200MS_EINVAL, "maxsim_rowm: B1 needs the per-group token counts");
    if (int e = reserve(h, h->b1_q_i8, size_t(n_q_rows) * 128 + 1024)) return e;
    if (int e = reserve(h, h->b1_tok_const, size_t(n_q_rows) * 4)) return e;
    uint8_t* q_i8 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(h->b1_q_i8.p) + 1023) & ~uintptr_t(1023));
    int32_t* tc = static_cast<int32_t*>(h->b1_tok_const.p);
    rowm_query_expand_kernel<<<(n_q_rows * 4 + 255) / 256, 256, 0, s>>>(static_cast<const uint32_t*>(q_packed), ntok_dev, n_q_rows,
                                                                       reinterpret_cast<uint4*>(q_i8), tc);
    h->launches++;
    if (int e = check_cuda(h, cudaGetLastError(), "launch rowm_query_expand")) return e;
    q_rows = q_i8;
    q_dtype = B200MS_I8;
    tok_const = tc;
  } else if (!c.has_tmap) {
    return set_error(h, B200MS_ESTATE, "score: corpus has no TMA descriptor");
  }
  const CUtensorMap* tq;  // the query is the N operand: a 32*NG-row box
  if (int e = query_tmap(h, q_rows, q_dtype, n_q_rows, 32 * ng, &tq)) return e;
  switch (c.dtype) {
    case B200MS_BF16:
      return ng == 1 ? launch_rowm_one<0, 1>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s)
                     : launch_rowm_one<0, 2>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s);
    case B200MS_I8:
      return ng == 1 ? launch_rowm_one<1, 1>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s)
                     : launch_rowm_one<1, 2>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s);
    case B200MS_F8:
      return ng == 1 ? launch_rowm_one<2, 1>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s)
                     : launch_rowm_one<2, 2>(h, *tq, tok_const, n_groups_real, clamp_bits, group_scores, ld, s);
    case B200MS_B1:  // one group only: with 640 threads the two-group epilogue does not fit the 96-register budget
      if (ng != 1) return set_error(h, B200MS_EINVAL, "maxsim_rowm: sign-bit corpora take one query group");
      return launch_rowm_one<3, 1>(h, *tq, tok_const, n_groups_real, nullptr, group_scores, ld, s);
    default:
      return set_error(h, B200MS_ESTATE, "score: corpus dtype has no row-major-M scorer");
  }
}

}  // namespace bms
