// common.cuh -- handle layout, error plumbing and kernel-launcher prototypes shared by the .cu files.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/b200ms.h"

namespace bms {

constexpr int kDim = B200MS_DIM;
constexpr int kGroup = B200MS_ROW_GROUP;  // 32 rows: padding granule of pages and queries ("chunk")
constexpr int kTileN = 128;               // patch rows per MMA tile (4 chunks)
constexpr int kTileM = 128;               // query rows per MMA tile (4 groups)
constexpr int kRowmMaxGroups = 2;         // maxsim_rowm.cu (patch rows as the M operand): scans of <= 2 query groups

struct DeviceBuf {  // grow-only device scratch
  void* p = nullptr;
  size_t cap = 0;
};
struct PinnedBuf {  // grow-only pinned + device-mapped host block (cudaHostAlloc)
  void* p = nullptr;
  size_t cap = 0;
};
struct DeviceGuard {  // switch to the handle's device for the duration of a call
  int prev = -1;
  explicit DeviceGuard(int dev);
  ~DeviceGuard();
};
// candidate list(s) of a rerank call: ids (device int64, -1 = unused slot); per_query = 0: one list of n_cand ids shared by
// every query; 1: [n_q, roundup(n_cand,32)] -- one list per query
struct SearchCand {
  const int64_t* ids = nullptr;
  int n_cand = 0;
  int per_query = 0;
};
struct Comm;  // comm.cu: NCCL communicator + the exchange pipeline of the sharded search

// Which chunk ranges a scoring launch walks.  Full scan: the corpus' own unit plan, scores indexed by page id.
// Candidate ("slot") mode: unit j = the chunk range of candidate page j, scores indexed by j.
struct UnitPlan {
  const int32_t* start = nullptr;
  const int32_t* end = nullptr;
  int n_units = 0;
  int slot_mode = 0;
  // zero_pad_compat: bit i set = page i (slot_mode: candidate slot i) is shorter than the longest page of its scoring
  // batch, so its per-token maxima are clamped at 0 like the reference's zero padding does; NULL = clean MaxSim
  const uint32_t* clamp_bits = nullptr;
};

struct Corpus {
  const void* rows = nullptr;
  int dtype = -1;
  int64_t n_pages = 0;
  int64_t n_rows = 0;    // padded rows
  int64_t n_chunks = 0;  // n_rows / 32
  int n_units = 0;
  CUtensorMap tmap;      // [n_rows,128] view, box = {128 B, kTileN rows}, SWIZZLE_128B (BF16 / I8 only)
  bool has_tmap = false;
  bool has_empty = false;  // some page has zero rows (its score is the memset 0)
  int64_t clamp_batch = 0;  // zero_pad_compat batch size the full-scan clamp bitmask (b200ms::clamp_pages) was built for
};

// Tensor maps of the query rows of the scoring launches (query_tmap), keyed on everything such a map encodes.  A map
// depends on nothing else, so an entry never goes stale; a miss re-encodes into the oldest slot.
struct QueryTmaps {
  struct Entry {
    const void* base = nullptr;
    int dtype = -1;  // -1: empty slot
    int64_t rows = 0;
    int box_rows = 0;
    CUtensorMap map;
  };
  static constexpr int kSlots = 4;  // a scoring call needs one map; a miss costs one host-side encode
  Entry slot[kSlots];
  int next = 0;  // slot the next miss fills
};

}  // namespace bms

struct b200ms {
  int device = 0;
  int num_sms = 0;
  std::string err;
  bms::Corpus corpus;
  // device metadata of the attached corpus
  bms::DeviceBuf chunk_page;   // int32 [n_chunks]   page index of every 32-row chunk
  bms::DeviceBuf unit_start;   // int32 [n_units+1]  first chunk of every work unit (page aligned)
  bms::DeviceBuf page_start;   // int64 [n_pages+1]  first padded row of every page   (B1 kernel, pack)
  bms::DeviceBuf page_len;     // int32 [n_pages]    TRUE row count of every page (zero_pad_compat, FDE from packed rows)
  bms::DeviceBuf clamp_pages;  // uint32 words: zero_pad_compat clamp bit per page (full scan), built lazily
  bms::DeviceBuf clamp_slots;  // uint32 words: clamp bit per candidate slot (rerank), rebuilt per call
  std::vector<int32_t> page_len_host;
  // scratch for pack / search
  bms::DeviceBuf meta, meta_b;  // per-call metadata block of a search (one upload) / of a pack call
  bms::DeviceBuf q_raw, q_packed, scores, mask, mask_index, out_all;
  bms::PinnedBuf stage;         // host entry points: [metadata | query rows | results], mapped into the device address space
  bms::DeviceBuf topk_keys, topk_ids;  // first-level (per-slice) top-k candidates
  bms::DeviceBuf b1_q_i8, b1_tok_const;  // tensor-core 1-bit scorer: +-1 int8 query tiles and per-token constants
  bms::DeviceBuf cand_pad;  // batched rerank: per-query candidate lists re-laid out with a 32-slot-aligned stride
  bms::DeviceBuf cand_start, cand_end, cand_mask;  // candidate (rerank) mode: per-slot chunk ranges, valid-slot bitmask
  bms::DeviceBuf fde_simhash, fde_ams_index, fde_ams_sign, fde_tmp;  // FDE configuration (device copies) + scratch
  bms::DeviceBuf fde_q_bf16;                      // scan: query FDEs split into bf16 hi/lo rows (tcgen05 B operand)
  bms::DeviceBuf fde_final_index, fde_final_sign; // optional final count-sketch projection (final_projection_dimension)
  int fde_dim = 0, fde_reps = 0, fde_ksim = 0, fde_proj = 0;
  int fde_inner_dim = 0;   // reps * 2^ksim * proj (before the optional final projection)
  int fde_fill_empty = 0;  // fill_empty_partitions (documents): empty partition <- projection of the nearest point
  int fde_gemm = 1;        // 1: scan on tcgen05 (fde_scan_umma_kernel) when the shape allows, 0: SIMT scan
  float fde_scale = 1.f;
  int zero_copy = 1;       // host entry points: small calls read queries / write results through mapped pinned memory
  bms::Comm* comm = nullptr;
  cudaStream_t stream = nullptr;  // internal stream for *_host entry points
  // ring of CUDA-event pairs bracketing the scoring kernels of the most recent b200ms_score / search calls
  static constexpr int kEvRing = 256;
  cudaEvent_t ev0[kEvRing] = {}, ev1[kEvRing] = {};
  int64_t ev_count = 0;  // scoring calls recorded since creation / last reset
  int64_t launches = 0;
  int64_t unit_rows = 4096;
  int max_ctas = 0;
  int b1_tensor = 2;  // 1-bit corpora: 0 = POPC kernel, 1 = tcgen05 kernel (bits expanded to {0,1} int8 in smem), 2 = auto
  int pair_cta = 2;   // CTA-pair kernels (cta_group::2, maxsim_umma_pair.cu): 0 off, 1 for passes of >= 3 query tiles, 2 (default) also for 2 tiles
  int pair_clusters = -1;  // co-resident CTA pairs the device reports for the pair kernel (-1: not queried yet)
  int zero_pad_batch = 0;  // > 0: reproduce score_multi_vector's zero-padding quirk with this batch size (128 upstream)
  bms::QueryTmaps query_tmaps;
  int rowm = 1;  // option "rowm": full scans of <= kRowmMaxGroups query groups run on maxsim_rowm_kernel (0: query-as-M kernels)
  // CUDA graphs of the small zero-copy host search (pack -> score -> top-k): key -> executable graph
  struct HostGraph {
    uint64_t key = 0;
    uint64_t generation = 0;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    int seen = 0;  // uses of this key so far; the graph is captured on the second one (buffers are warm by then)
    uint64_t last_use = 0;
  };
  std::vector<HostGraph> host_graphs;
  uint64_t generation = 0;   // bumped whenever a scratch buffer moves, the corpus is re-attached or an option changes
  uint64_t graph_clock = 0;
  int host_graph = 1;        // option "host_graph": replay small unmasked host searches as one CUDA graph
  bool capturing = false;    // inside stream capture: no event timing, no allocation

};

namespace bms {

int set_error(b200ms_t* h, int code, const std::string& msg);
int check_cuda(b200ms_t* h, cudaError_t e, const char* what);
int reserve(b200ms_t* h, DeviceBuf& b, size_t bytes);
int upload(b200ms_t* h, DeviceBuf& b, const void* src, size_t bytes, cudaStream_t s);
int reserve_pinned(b200ms_t* h, PinnedBuf& b, size_t bytes);
// Raise cudaFuncAttributeMaxDynamicSharedMemorySize when static + dynamic shared memory passes the 48 KB default; process-global
// raise-only table per (device, kernel) -- the attribute belongs to the function, not to the handle
int ensure_smem(b200ms_t* h, const void* kernel, int smem, const char* what);
int make_tmap_rows(b200ms_t* h, CUtensorMap* out, const void* base, int dtype, int64_t n_rows, int box_rows,
                   int64_t row_bytes = 0);
// make_tmap_rows of query rows (default row bytes) through the handle's QueryTmaps; a later call may re-encode *out
int query_tmap(b200ms_t* h, const void* base, int dtype, int64_t n_rows, int box_rows, const CUtensorMap** out);
void comm_teardown(b200ms_t* h);
// pack -> score -> top-k on stream s (api.cu); meta_in_place / meta_host_block: see the definition
int search_core(b200ms_t* h, const void* q_src, int src_dtype, const int32_t* q_lens, int n_q, int k,
                const uint32_t* allow_dev, float i8_q_scale, float score_scale, int64_t id_base, float* ts, int64_t* ti,
                int32_t* tc, cudaStream_t s, const SearchCand* cand, const int32_t* mask_index_dev, int64_t mask_stride,
                const void* meta_in_place, const void* meta_host_block);

// kernel launchers (each returns a b200ms error code and bumps h->launches)
int launch_score_umma(b200ms_t* h, const UnitPlan* plan, const void* q_packed, int n_groups_real, void* group_scores,
                      int64_t ld, cudaStream_t s, int m_tile = -1);
constexpr int B200MS_EUNSUPPORTED_PAIR = -100;  // internal: pair kernel cannot be scheduled on this device
int launch_score_umma_pair(b200ms_t* h, const UnitPlan& up, const CUtensorMap& tq, int nm, int m_tile_base,
                           int n_groups_real, void* scores, int64_t ld, cudaStream_t s);
int launch_score_b1(b200ms_t* h, const int64_t* cand_ids, int64_t n_cand, const void* q_packed, int n_groups,
                    const int32_t* group_ntok_dev, void* group_scores, int64_t ld, cudaStream_t s, int g_lo, int g_hi);
int launch_pad_cands(b200ms_t* h, const int64_t* src, int n_cand, int n_lists, int64_t stride, int64_t* dst, cudaStream_t s);
int launch_clamp_slots(b200ms_t* h, const int64_t* cand_ids, int n_cand, int n_lists, int64_t list_stride, int batch,
                       uint32_t* clamp_bits, cudaStream_t s);
int launch_score_b1_umma(b200ms_t* h, const void* q_bits, const int32_t* group_ntok_dev, int n_groups_real,
                         void* group_scores, int64_t ld, cudaStream_t s);
int launch_score_rowm(b200ms_t* h, const void* q_packed, int n_groups_real, const int32_t* ntok_dev, const uint32_t* clamp_bits,
                      void* group_scores, int64_t ld, cudaStream_t s);
int launch_cand_units(b200ms_t* h, const int64_t* cand_ids, int n_cand, int32_t* unit_start, int32_t* unit_end,
                      uint32_t* slot_mask, cudaStream_t s);
int launch_hamming_batch(b200ms_t* h, const void* q, const void* cand, int64_t n, uint32_t* out, cudaStream_t s);
int launch_sign_pack(b200ms_t* h, const void* x, int src_dtype, int64_t rows, uint8_t* out, cudaStream_t s);
int launch_chunk_page(b200ms_t* h, const int64_t* page_start_dev, int64_t n_pages, int32_t* chunk_page, cudaStream_t s);
int launch_pack_rows(b200ms_t* h, const void* src, int src_dtype, const int64_t* src_start_dev,
                     const int64_t* dst_start_dev, int64_t n_items, int64_t dst_rows, int pad_mode, void* dst,
                     int dst_dtype, float i8_scale, cudaStream_t s);
int launch_topk(b200ms_t* h, const void* group_scores, int score_dtype, int64_t n_pages, int64_t ld,
                const int32_t* group_offsets_dev, int n_q, const uint32_t* allow_mask, int k, float scale,
                int64_t id_base, const int64_t* id_map, float* top_scores, int64_t* top_ids, int32_t* top_counts,
                cudaStream_t s, const int32_t* mask_index = nullptr, int64_t mask_stride = 0, int64_t q_stride = 0);
// merge straight from the all-gathered exchange layout: gathered = world blocks of [n_q*k int64 ids | n_q*k f32 scores]
int launch_merge_gathered(b200ms_t* h, const void* gathered, int world, int n_q, int k, float* top_scores, int64_t* top_ids,
                          int32_t* top_counts, cudaStream_t s);
int launch_fde_encode(b200ms_t* h, const void* rows, int src_dtype, const int64_t* item_start_dev, int n_items,
                      int is_document, float* out, cudaStream_t s, const int32_t* item_len_dev = nullptr);
int launch_fde_finalize(b200ms_t* h, const float* fde, int64_t n, void* out_rows, float* inv_norm, cudaStream_t s);
int launch_fde_scan(b200ms_t* h, const void* F, const float* inv_norm, int64_t n_pages, const float* q_fde, int n_q,
                    float* scores, int64_t ld, cudaStream_t s);
int launch_merge_topk(b200ms_t* h, const float* cand_scores, const int64_t* cand_ids, int n_q, int m, int k,
                      float* top_scores, int64_t* top_ids, int32_t* top_counts, cudaStream_t s);

}  // namespace bms
