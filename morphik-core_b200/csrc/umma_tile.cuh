// umma_tile.cuh -- tile geometry, pipeline pieces and accumulator helpers shared by the query-as-M tcgen05 MaxSim kernels
// (maxsim_umma.cu: one CTA per SM; maxsim_umma_pair.cu: CTA pairs, cta_group::2; maxsim_b1_umma.cu: 1-bit rows).  The
// lone-query kernel (maxsim_rowm.cu) also uses the teardown and launch_persistent, the FDE scan (fde.cu) the CTA layout and
// lifetime pieces and launch_persistent.
#pragma once
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace bms {

constexpr int kNumAccum = 4;                     // TMEM accumulators, kTileN fp32 columns each (4*128 = 512)
constexpr uint32_t kSubtileBytes = 128 * 128;    // 128 rows x 128 B (one swizzle-128B panel)
constexpr uint32_t kSmemLimit = 232448;          // 227 KB opt-in maximum per CTA
constexpr uint32_t kBarrierBytes = 2048;         // mbarriers + TMEM slot

// KIND 0: bf16 rows (256 B = two 128 B K-panels), kind::f16, fp32 accumulators
// KIND 1: int8 rows (128 B = one panel),           kind::i8,  int32 accumulators (exact)
// KIND 2: fp8 e4m3 rows (128 B = one panel),       kind::f8f6f4, fp32 accumulators
// Every tcgen05.mma step consumes 32 B of K per row.
template <int KIND>
struct Kind {
  static constexpr int kPanels = KIND == 0 ? 2 : 1;
  static constexpr uint32_t kTileBytes = kPanels * kSubtileBytes;
  static constexpr int kPanelElems = KIND == 0 ? 64 : 128;  // TMA x-coordinate step per panel (elements)
  static constexpr int kKSteps = KIND == 0 ? 8 : 4;         // tcgen05.mma K steps per 128-d row
  static constexpr int kMaxNM = KIND == 0 ? 4 : 8;          // query tiles one CTA can keep resident in shared memory
  using Acc = typename std::conditional<KIND == 1, int, float>::type;
};

// corpus dtype (include/b200ms.h) -> kernel KIND, or -1
__host__ __device__ constexpr int kind_of_dtype(int dtype) {
  return dtype == B200MS_BF16 ? 0 : dtype == B200MS_I8 ? 1 : dtype == B200MS_F8 ? 2 : -1;
}

__device__ __forceinline__ float acc_from_bits(uint32_t v, float) { return __uint_as_float(v); }
__device__ __forceinline__ int acc_from_bits(uint32_t v, int) { return static_cast<int>(v); }
__device__ __forceinline__ float acc_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ int acc_max(int a, int b) { return max(a, b); }

// max over the 32 columns a thread holds for one chunk (two independent chains for ILP)
__device__ __forceinline__ float chunk_max_f(const uint32_t (&v)[32]) {
  float a = __uint_as_float(v[0]);
  float b = __uint_as_float(v[1]);
#pragma unroll
  for (int i = 2; i < 30; i += 4) {
    a = fmax3(a, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
    b = fmax3(b, __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
  }
  a = fmax3(a, __uint_as_float(v[30]), __uint_as_float(v[31]));
  return fmaxf(a, b);
}
__device__ __forceinline__ int chunk_max_i(const uint32_t (&v)[32]) {
  int a = int(v[0]), b = int(v[1]);
#pragma unroll
  for (int i = 2; i < 30; i += 4) {
    a = imax3(a, int(v[i]), int(v[i + 1]));
    b = imax3(b, int(v[i + 2]), int(v[i + 3]));
  }
  a = imax3(a, int(v[30]), int(v[31]));
  return max(a, b);
}
// (Round 2 tried the int32 accumulators on the FLOAT min/max datapath -- bit patterns of non-negative ints below 0x7f800000 order
// like floats, with an integer redo when the float maximum came back negative / NaN.  Exact, but it bought nothing in the batch
// regime (TMEM-drain-bound, 6.16 vs 6.24 ms) and cost 37 % for ONE query, where a single warp's dependent max chain is the
// critical path: 1.42 ms integer vs 1.95 ms float at 65 536 pages, profiles/r02/ab_epilogue_variants.jsonl.  Integer it is.)
template <typename Acc>
__device__ __forceinline__ Acc chunk_max(const uint32_t (&v)[32]) {
  if constexpr (std::is_same<Acc, float>::value) {
    return chunk_max_f(v);
  } else {
    return chunk_max_i(v);
  }
}

// zero_pad_compat (option "zero_pad_compat"): colpali_engine's score_multi_vector pads every batch of pages with zero rows
// up to the longest page of the batch and lets them take part in the max (transformers port processing_colpali.py:350-362),
// so a page shorter than its batch's longest scores sum_t max(true max_t, 0).  clamp_bits bit i = "page (or candidate slot) i
// is shorter than the longest of its batch"; NULL = clean MaxSim (the default).
template <typename Acc>
__device__ __forceinline__ Acc clamp_token_max(const uint32_t* __restrict__ clamp_bits, int idx, Acc rm) {
  if (clamp_bits != nullptr && ((__ldg(clamp_bits + (idx >> 5)) >> (idx & 31)) & 1u)) return acc_max(rm, Acc(0));
  return rm;
}

// ---------------------------------------------------------------------------------------------- CTA layout and lifetime
// Dynamic shared memory: [1024-aligned] resident query tiles | num_stages patch tiles | kBarrierBytes of barriers.
struct TileSmem {
  uint8_t* q;
  uint8_t* st;
  uint64_t* full;    // [num_stages] producer -> MMA
  uint64_t* empty;   // [num_stages] MMA -> producer
  uint64_t* tfull;   // [accumulators] MMA -> epilogue
  uint64_t* tempty;  // [accumulators] epilogue -> MMA
  uint64_t* qfull;   // query tiles landed
  uint32_t* tmem_slot;
};

__device__ __forceinline__ TileSmem carve_tile_smem(uint8_t* raw, uint32_t q_bytes, uint32_t tile_bytes, int num_stages) {
  TileSmem sm;
  sm.q = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
  sm.st = sm.q + q_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm.st + size_t(num_stages) * tile_bytes);
  sm.full = bars;
  sm.empty = bars + 16;
  sm.tfull = bars + 32;
  sm.tempty = bars + 40;
  sm.qfull = bars + 48;
  sm.tmem_slot = reinterpret_cast<uint32_t*>(bars + 56);
  return sm;
}

// Thread 0 prefetches the tensor maps (tmap_b may be null) and initialises the barriers, warp 2 allocates all 512 TMEM
// columns, and the CTA (PAIR: the cluster) synchronises so both are visible before any arrive or TMA signal.
template <bool PAIR>
__device__ __forceinline__ uint32_t tile_prologue(const TileSmem& sm, int warp, const CUtensorMap* tmap_a,
                                                  const CUtensorMap* tmap_b, int num_stages, uint32_t full_count, int n_accum,
                                                  uint32_t tempty_count) {
  if (threadIdx.x == 0) {
    prefetch_tmap(tmap_a);
    if (tmap_b != nullptr) prefetch_tmap(tmap_b);
    for (int i = 0; i < num_stages; ++i) {
      mbar_init(&sm.full[i], full_count);
      mbar_init(&sm.empty[i], 1);
    }
    for (int i = 0; i < n_accum; ++i) {
      mbar_init(&sm.tfull[i], 1);
      mbar_init(&sm.tempty[i], tempty_count);
    }
    mbar_init(sm.qfull, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (PAIR) tmem_alloc_512_pair(sm.tmem_slot);
    else tmem_alloc_512(sm.tmem_slot);
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  return *sm.tmem_slot;
}

// Nobody exits (or frees TMEM) while another warp -- PAIR: the partner CTA -- can still touch shared memory or TMEM.
template <bool PAIR>
__device__ __forceinline__ void tile_teardown(int warp, uint32_t tmem_base) {
  if constexpr (PAIR) __syncwarp();
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (PAIR) tmem_dealloc_512_pair(tmem_base);
    else tmem_dealloc_512(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------- MMA issue
// One 128-deep contraction into d_tmem: K::kKSteps tcgen05.mma of 32 B of K each, four per 128 B panel; ad / bd describe
// the first panel of the A / B tile.  PAIR issues the cta_group::2 form.
template <int KIND, bool PAIR = false>
__device__ __forceinline__ void umma_tile(uint32_t d_tmem, uint64_t ad, uint64_t bd, uint32_t idesc) {
#pragma unroll
  for (int ks = 0; ks < Kind<KIND>::kKSteps; ++ks) {
    const uint32_t off = ((ks >> 2) * kSubtileBytes + (ks & 3) * 32) >> 4;
    if constexpr (PAIR) umma2_ss<KIND>(d_tmem, ad + off, bd + off, idesc, ks != 0);
    else umma_ss<KIND>(d_tmem, ad + off, bd + off, idesc, ks != 0);
  }
}

// ---------------------------------------------------------------------------------------------- epilogue
// Hand an accumulator back to the MMA warp; release() is the arrive on tempty (local, or on the leader CTA's barrier).
template <typename Release>
__device__ __forceinline__ void release_accum(Release&& release) {
  tc_fence_before();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) release();
}

// Drain the 128 columns of one accumulator in this warp's lane quadrant: cm[j] = the thread's maximum over chunk j.  Two
// loads stay in flight, and the accumulator is released as soon as the last one has landed, before the last two maxima.
template <typename Acc, typename Release>
__device__ __forceinline__ void drain_accum(uint32_t taddr, Acc (&cm)[4], Release&& release) {
  uint32_t va[32], vb[32];
  tmem_ld_32x32(taddr, va);
  tmem_ld_32x32(taddr + 32, vb);
  tmem_ld_wait();
  cm[0] = chunk_max<Acc>(va);
  cm[1] = chunk_max<Acc>(vb);
  tmem_ld_32x32(taddr + 64, va);
  tmem_ld_32x32(taddr + 96, vb);
  tmem_ld_wait();
  release_accum(release);
  cm[2] = chunk_max<Acc>(va);
  cm[3] = chunk_max<Acc>(vb);
}

// pg[j] = page of chunk cb + j of a tile, or -1 past the unit's last chunk c1
__device__ __forceinline__ void tile_pages(const int32_t* __restrict__ chunk_page, int cb, int c1, int (&pg)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) pg[j] = (cb + j < c1) ? __ldg(chunk_page + cb + j) : -1;
}

// One closed (group, page) run of the bf16 / int8 / fp8 kernels: zero_pad_compat clamp, 32-token sum, lane 0 stores column o.
template <typename Acc>
__device__ __forceinline__ void store_group_score(Acc* __restrict__ group_scores, int64_t ld, int group, int o,
                                                  const uint32_t* __restrict__ clamp_bits, Acc rm) {
  const Acc s = warp_sum(clamp_token_max(clamp_bits, o, rm));
  if ((threadIdx.x & 31) == 0) group_scores[int64_t(group) * ld + o] = s;
}

// The running per-token max of one query group over its open page.  Units hold whole pages, so a page closes either at a
// page change inside fold() or at the unit's end (flush()).  emit(page, rm) writes one closed page: the kernel's output
// index, clamp, 32-token warp sum and lane-0 store.
template <typename Acc>
struct PageRun {
  Acc rm;
  int cp = -1;  // open page, -1: none

  template <typename Emit>
  __device__ __forceinline__ void fold(const int (&pg)[4], const Acc (&cm)[4], Emit&& emit) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (pg[j] < 0) continue;  // chunk belongs to the next unit
      if (pg[j] != cp) {
        if (cp >= 0) emit(cp, rm);
        cp = pg[j];
        rm = cm[j];
      } else {
        rm = acc_max(rm, cm[j]);
      }
    }
  }
  template <typename Emit>
  __device__ __forceinline__ void flush(Emit&& emit) {
    if (cp >= 0) emit(cp, rm);
    cp = -1;
  }
};

// One stream of work units u, u + stride, ... walked one 128-row tile (4 chunks) at a time, skipping empty units.
struct UnitWalk {
  int u, stride, c0, c1, t, n_tiles;
  __device__ __forceinline__ void load(const int32_t* us, const int32_t* ue, int n_units) {
    n_tiles = 0;
    while (u < n_units) {
      c0 = __ldg(us + u);
      c1 = __ldg(ue + u);
      n_tiles = (c1 - c0 + 3) >> 2;
      if (n_tiles > 0) break;
      u += stride;
    }
    t = 0;
  }
  __device__ __forceinline__ void init(int v, int stride_, const int32_t* us, const int32_t* ue, int n_units) {
    u = v;
    stride = stride_;
    load(us, ue, n_units);
  }
  __device__ __forceinline__ bool valid(int n_units) const { return u < n_units; }
  __device__ __forceinline__ int chunk() const { return c0 + 4 * t; }  // first chunk of the current tile
  __device__ __forceinline__ void next(const int32_t* us, const int32_t* ue, int n_units) {
    if (++t == n_tiles) {
      u += stride;
      load(us, ue, n_units);
    }
  }
};

// ---------------------------------------------------------------------------------------------- host side
// Stage ring of a kernel whose dynamic shared memory is [1024-aligned] resident_bytes | stages x tile_bytes | kBarrierBytes:
// as many stages as fit the 227 KB opt-in, at most max_stages, at least 2.  tile_bytes = 0: the stages hold no shared memory
// (maxsim_rowm_kernel<3> keeps its A tiles in TMEM) and there are max_stages of them.  Raises the kernel's shared-memory limit.
static int size_stage_ring(b200ms_t* h, const void* kern, const char* name, uint32_t resident_bytes, uint32_t tile_bytes,
                           int max_stages, int* stages, uint32_t* smem) {
  int n = tile_bytes ? int((kSmemLimit - 1024 /*align*/ - kBarrierBytes - resident_bytes) / tile_bytes) : max_stages;
  if (n > max_stages) n = max_stages;
  if (n < 2) return set_error(h, B200MS_EINVAL, std::string(name) + ": not enough shared memory for 2 stages");
  *stages = n;
  *smem = 1024 + resident_bytes + uint32_t(n) * tile_bytes + kBarrierBytes;
  return ensure_smem(h, kern, int(*smem), name);
}

// Persistent one-CTA launch on a size_stage_ring ring, grid = one CTA per SM (or max_ctas), at most one per unit.
// num_stages is the kernel's last argument.
template <typename... Params, typename... Args>
static int launch_persistent(b200ms_t* h, void (*kern)(Params...), const char* name, int threads, uint32_t resident_bytes,
                             uint32_t tile_bytes, int max_stages, int n_units, cudaStream_t s, Args... args) {
  int stages;
  uint32_t smem;
  if (int e = size_stage_ring(h, reinterpret_cast<const void*>(kern), name, resident_bytes, tile_bytes, max_stages, &stages,
                              &smem))
    return e;
  int grid = h->max_ctas > 0 ? h->max_ctas : h->num_sms;
  if (grid > n_units) grid = n_units;
  if (grid < 1) return B200MS_OK;
  kern<<<grid, threads, smem, s>>>(args..., stages);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), name);
}

}  // namespace bms
