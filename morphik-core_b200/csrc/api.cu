// api.cu -- the extern "C" surface declared in include/b200ms.h: handle management, corpus attachment
// (chunk table, work-unit plan, TMA descriptor), query packing and the fused search entry points.
// Host-side C++ only orchestrates; all arithmetic on embeddings happens in the CUDA kernels.
// (Multi-GPU entry points -- NCCL communicator, all-gather of top-k lists, pipelined sharded search -- live in comm.cu.)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace bms {

static std::mutex g_err_mu;
static std::string g_err;

int set_error(b200ms_t* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  std::lock_guard<std::mutex> lk(g_err_mu);
  g_err = msg;
  return code;
}

int check_cuda(b200ms_t* h, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return B200MS_OK;
  return set_error(h, B200MS_ECUDA, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}

int reserve(b200ms_t* h, DeviceBuf& b, size_t bytes) {
  if (bytes <= b.cap) return B200MS_OK;
  if (h) {
    if (h->capturing) return set_error(h, B200MS_ESTATE, "scratch buffer would grow inside a graph capture");
    h->generation++;  // captured graphs hold the old address
  }
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  size_t want = bytes + bytes / 4;
  want = (want + 1023) & ~size_t(1023);
  if (cudaMalloc(&b.p, want) != cudaSuccess) {
    cudaGetLastError();
    want = (bytes + 1023) & ~size_t(1023);
    if (cudaError_t e = cudaMalloc(&b.p, want); e != cudaSuccess) {
      b.p = nullptr;
      cudaGetLastError();
      return set_error(h, B200MS_ENOMEM, "cudaMalloc of " + std::to_string(want) + " scratch bytes failed");
    }
  }
  b.cap = want;
  return B200MS_OK;
}

int reserve_pinned(b200ms_t* h, PinnedBuf& b, size_t bytes) {
  if (bytes <= b.cap) return B200MS_OK;
  if (h) h->generation++;
  if (b.p) cudaFreeHost(b.p);
  b.p = nullptr;
  b.cap = 0;
  const size_t want = ((bytes + bytes / 4) + 4095) & ~size_t(4095);
  // cudaHostAllocMapped: with unified addressing the same pointer is valid in kernels (zero-copy reads / writes over PCIe)
  if (cudaError_t e = cudaHostAlloc(&b.p, want, cudaHostAllocMapped | cudaHostAllocPortable); e != cudaSuccess) {
    b.p = nullptr;
    cudaGetLastError();
    return set_error(h, B200MS_ENOMEM, "cudaHostAlloc of " + std::to_string(want) + " pinned bytes failed");
  }
  b.cap = want;
  return B200MS_OK;
}

// MaxDynamicSharedMemorySize is a property of the FUNCTION in the device's context, shared by every handle of the process:
// it must only ever be raised.  (A per-handle cache let a second handle "set" a small value for the merge kernel and thereby
// LOWER the limit a first handle relied on -- its next large merge then failed with cudaErrorInvalidValue.)  Launches that fit
// the 48 KB default need no call at all.
int ensure_smem(b200ms_t* h, const void* kernel, int smem, const char* what) {
  if (smem <= 16 * 1024) return B200MS_OK;  // static + dynamic cannot pass the 48 KB default below this
  struct Entry {
    int static_bytes;
    int raised;  // largest MaxDynamicSharedMemorySize set so far (0 = never set)
  };
  static std::mutex mu;
  static std::unordered_map<uint64_t, Entry> table;  // (device, kernel)
  const uint64_t key = (uint64_t(uint32_t(h ? h->device : 0)) << 56) ^ uint64_t(reinterpret_cast<uintptr_t>(kernel));
  std::lock_guard<std::mutex> lk(mu);
  auto it = table.find(key);
  if (it == table.end()) {
    cudaFuncAttributes fa;
    if (int e = check_cuda(h, cudaFuncGetAttributes(&fa, kernel), what)) return e;
    it = table.emplace(key, Entry{int(fa.sharedSizeBytes), 0}).first;
  }
  Entry& en = it->second;
  // the default limit (48 KB) covers the kernel's STATIC shared memory as well as the dynamic request
  if (en.raised == 0 && smem + en.static_bytes <= 48 * 1024) return B200MS_OK;
  if (en.raised >= smem) return B200MS_OK;
  if (int e = check_cuda(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), what)) return e;
  en.raised = smem;
  return B200MS_OK;
}

int upload(b200ms_t* h, DeviceBuf& b, const void* src, size_t bytes, cudaStream_t s) {
  if (int e = reserve(h, b, bytes ? bytes : 16)) return e;
  if (bytes == 0) return B200MS_OK;
  return check_cuda(h, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, s), "upload metadata");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Resolved once per process, thread-safe (handles on different threads may attach corpora concurrently).
static EncodeTiledFn encode_fn(b200ms_t* h) {
  static std::once_flag once;
  static EncodeTiledFn fn = nullptr;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess && p) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    } else {
      cudaGetLastError();
    }
  });
  if (!fn) set_error(h, B200MS_ECUDA, "cuTensorMapEncodeTiled not available from the driver");
  return fn;
}

// [n_rows, row_bytes] row-major view; box = one 128-byte K panel x box_rows rows, 128-byte swizzle (what the UMMA
// K-major SWIZZLE_128B descriptor expects).  Out-of-range rows read as zero.  row_bytes is 256 for bf16 rows and 128 for
// the one-byte dtypes by default; the FDE matrix passes its own (fde_dim * 2).
int make_tmap_rows(b200ms_t* h, CUtensorMap* out, const void* base, int dtype, int64_t n_rows, int box_rows, int64_t row_bytes) {
  EncodeTiledFn fn = encode_fn(h);
  if (!fn) return B200MS_ECUDA;
  const bool bf16 = dtype == B200MS_BF16;
  if (row_bytes <= 0) row_bytes = bf16 ? 256 : 128;
  const cuuint64_t dims[2] = {cuuint64_t(bf16 ? row_bytes / 2 : row_bytes), cuuint64_t(n_rows > 0 ? n_rows : 1)};
  const cuuint64_t strides[1] = {cuuint64_t(row_bytes)};
  const cuuint32_t box[2] = {cuuint32_t(bf16 ? 64 : 128), cuuint32_t(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(out, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2,
                        const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(h, B200MS_ECUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(r)));
  return B200MS_OK;
}

int query_tmap(b200ms_t* h, const void* base, int dtype, int64_t n_rows, int box_rows, const CUtensorMap** out) {
  QueryTmaps& c = h->query_tmaps;
  for (QueryTmaps::Entry& en : c.slot) {
    if (en.base == base && en.dtype == dtype && en.rows == n_rows && en.box_rows == box_rows) {
      *out = &en.map;
      return B200MS_OK;
    }
  }
  QueryTmaps::Entry& en = c.slot[c.next];
  en.dtype = -1;
  if (int e = make_tmap_rows(h, &en.map, base, dtype, n_rows, box_rows)) return e;
  en.base = base;
  en.dtype = dtype;
  en.rows = n_rows;
  en.box_rows = box_rows;
  c.next = (c.next + 1) % QueryTmaps::kSlots;
  *out = &en.map;
  return B200MS_OK;
}

static bool corpus_dtype_ok(int d) { return d == B200MS_BF16 || d == B200MS_I8 || d == B200MS_B1 || d == B200MS_F8; }
static bool src_dtype_ok(int d) { return d == B200MS_F32 || d == B200MS_BF16; }

DeviceGuard::DeviceGuard(int dev) {
  cudaGetDevice(&prev);
  if (prev != dev) cudaSetDevice(dev);
}
DeviceGuard::~DeviceGuard() {
  int cur = -1;
  cudaGetDevice(&cur);
  if (prev >= 0 && cur != prev) cudaSetDevice(prev);
}

// ---- per-call metadata: ONE block (host-built) -> one upload, or read in place when the block is mapped pinned memory
struct SearchMeta {
  std::vector<uint8_t> host;  // [ss int64 (n_q+1) | ds int64 (n_q+1) | goff int32 (n_q+1) | ntok int32 (groups_padded)]
  size_t off_ss = 0, off_ds = 0, off_goff = 0, off_ntok = 0;
  int64_t rows = 0, groups = 0, groups_padded = 0;
  std::vector<int32_t> goff;
};

static void build_search_meta(const int32_t* q_lens, int n_q, SearchMeta* m) {
  const int64_t groups = b200ms_query_groups(q_lens, n_q);
  m->groups = groups;
  m->groups_padded = (groups + 3) & ~int64_t(3);
  const size_t n1 = size_t(n_q) + 1;
  m->off_ss = 0;
  m->off_ds = n1 * 8;
  m->off_goff = 2 * n1 * 8;
  m->off_ntok = m->off_goff + ((n1 * 4 + 15) & ~size_t(15));
  m->host.assign(m->off_ntok + size_t(m->groups_padded > 0 ? m->groups_padded : 4) * 4, 0);
  int64_t* ss = reinterpret_cast<int64_t*>(m->host.data() + m->off_ss);
  int64_t* ds = reinterpret_cast<int64_t*>(m->host.data() + m->off_ds);
  int32_t* goff = reinterpret_cast<int32_t*>(m->host.data() + m->off_goff);
  int32_t* ntok = reinterpret_cast<int32_t*>(m->host.data() + m->off_ntok);
  ss[0] = ds[0] = 0;
  goff[0] = 0;
  for (int i = 0; i < n_q; ++i) {
    const int64_t len = q_lens[i] > 0 ? q_lens[i] : 0;
    ss[i + 1] = ss[i] + len;
    ds[i + 1] = ds[i] + b200ms_padded_len(len);
    goff[i + 1] = int32_t(ds[i + 1] / kGroup);
    int64_t left = len;
    for (int g = goff[i]; g < goff[i + 1]; ++g) {
      ntok[g] = int32_t(left > kGroup ? kGroup : left);
      left -= ntok[g];
    }
  }
  m->rows = ss[n_q];
  m->goff.assign(goff, goff + n1);
}

}  // namespace bms

using namespace bms;

#define B200MS_API extern "C" __attribute__((visibility("default")))

B200MS_API int b200ms_version(void) { return B200MS_VERSION; }

B200MS_API int b200ms_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

B200MS_API const char* b200ms_last_error(const b200ms_t* h) {
  if (h) return h->err.c_str();
  std::lock_guard<std::mutex> lk(g_err_mu);
  return g_err.c_str();
}

B200MS_API int b200ms_create(int device, b200ms_t** out) {
  if (!out) return set_error(nullptr, B200MS_EINVAL, "create: out is NULL");
  *out = nullptr;
  int n = 0;
  if (cudaError_t e = cudaGetDeviceCount(&n); e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return set_error(nullptr, B200MS_ECUDA, "create: no CUDA device available (this library has no CPU fallback)");
  }
  if (device < 0 || device >= n) return set_error(nullptr, B200MS_EINVAL, "create: bad device index");
  DeviceGuard g(device);
  cudaDeviceProp prop;
  if (int e = check_cuda(nullptr, cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties")) return e;
  if (prop.major != 10) {
    return set_error(nullptr, B200MS_ECUDA, std::string("create: device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                                ", this library is built for sm_100a (B200) only");
  }
  b200ms_t* h = new b200ms_t();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  if (const char* e = getenv("B200MS_B1_TENSOR")) h->b1_tensor = atoi(e);
  if (const char* e = getenv("B200MS_PAIR_CTA")) h->pair_cta = atoi(e);
  if (const char* e = getenv("B200MS_ROWM")) h->rowm = atoi(e) != 0;
  if (const char* e = getenv("B200MS_ZERO_COPY")) h->zero_copy = atoi(e);
  if (const char* e = getenv("B200MS_UNIT_ROWS")) { if (atoll(e) > 0) h->unit_rows = atoll(e); }
  if (int e = check_cuda(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking), "cudaStreamCreate")) {
    delete h;
    return e;
  }
  for (int i = 0; i < b200ms_t::kEvRing; ++i) {
    if (cudaEventCreate(&h->ev0[i]) != cudaSuccess || cudaEventCreate(&h->ev1[i]) != cudaSuccess) {
      const int e = check_cuda(nullptr, cudaGetLastError(), "create: cudaEventCreate");
      b200ms_destroy(h);
      return e ? e : B200MS_ECUDA;
    }
  }
  *out = h;
  return B200MS_OK;
}

B200MS_API int b200ms_destroy(b200ms_t* h) {
  if (!h) return B200MS_OK;
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  comm_teardown(h);
  for (auto& g2 : h->host_graphs)
    if (g2.exec) cudaGraphExecDestroy(g2.exec);
  DeviceBuf* bufs[] = {&h->chunk_page, &h->unit_start, &h->page_start, &h->page_len, &h->clamp_pages, &h->clamp_slots,
                       &h->meta, &h->meta_b, &h->q_raw, &h->q_packed, &h->scores, &h->mask, &h->mask_index, &h->out_all,
                       &h->cand_pad, &h->cand_start, &h->cand_end, &h->cand_mask, &h->topk_keys, &h->topk_ids, &h->b1_q_i8, &h->b1_tok_const,
                       &h->fde_simhash, &h->fde_ams_index, &h->fde_ams_sign, &h->fde_tmp, &h->fde_q_bf16, &h->fde_final_index,
                       &h->fde_final_sign};
  for (DeviceBuf* b : bufs)
    if (b->p) cudaFree(b->p);
  if (h->stage.p) cudaFreeHost(h->stage.p);
  for (int i = 0; i < b200ms_t::kEvRing; ++i) {
    if (h->ev0[i]) cudaEventDestroy(h->ev0[i]);
    if (h->ev1[i]) cudaEventDestroy(h->ev1[i]);
  }
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return B200MS_OK;
}

B200MS_API int64_t b200ms_padded_len(int64_t len) { return len <= 0 ? 0 : (len + kGroup - 1) / kGroup * kGroup; }

B200MS_API int64_t b200ms_padded_rows(const int32_t* page_lens, int64_t n_pages) {
  int64_t t = 0;
  for (int64_t i = 0; i < n_pages; ++i) t += b200ms_padded_len(page_lens[i]);
  return t;
}

B200MS_API int64_t b200ms_row_bytes(int dtype) {
  switch (dtype) {
    case B200MS_F32: return 512;
    case B200MS_BF16: return 256;
    case B200MS_I8: return 128;
    case B200MS_F8: return 128;
    case B200MS_B1: return 16;
    default: return 0;
  }
}

B200MS_API int64_t b200ms_query_groups(const int32_t* q_lens, int n_q) {
  int64_t g = 0;
  for (int i = 0; i < n_q; ++i) g += (int64_t(q_lens[i] > 0 ? q_lens[i] : 0) + kGroup - 1) / kGroup;
  return g;
}

B200MS_API int64_t b200ms_launch_count(const b200ms_t* h) { return h ? h->launches : 0; }

B200MS_API int b200ms_set_tuning(b200ms_t* h, int64_t unit_rows, int max_ctas) {
  if (!h) return B200MS_EINVAL;
  if (unit_rows > 0) h->unit_rows = unit_rows;
  if (max_ctas >= 0) h->max_ctas = max_ctas;
  return B200MS_OK;
}

B200MS_API int b200ms_set_option(b200ms_t* h, const char* name, int64_t value) {
  if (!h || !name) return B200MS_EINVAL;
  const std::string n(name);
  if (n == "pair_cta" && value >= 0 && value <= 2) {
    h->pair_cta = int(value);
  } else if (n == "b1_tensor" && value >= 0 && value <= 2) {
    h->b1_tensor = int(value);
  } else if (n == "zero_pad_compat" && value >= 0 && value <= (int64_t(1) << 30)) {
    h->zero_pad_batch = int(value);
  } else if (n == "zero_copy" && value >= 0 && value <= 1) {
    h->zero_copy = int(value);
  } else if (n == "rowm" && value >= 0 && value <= 1) {
    h->rowm = int(value);
  } else if (n == "fde_gemm" && value >= 0 && value <= 1) {
    h->fde_gemm = int(value);
  } else if (n == "host_graph" && value >= 0 && value <= 1) {
    h->host_graph = int(value);
  } else if (n == "unit_rows" && value > 0) {
    h->unit_rows = value;
  } else if (n == "max_ctas" && value >= 0) {
    h->max_ctas = int(value);
  } else {
    return set_error(h, B200MS_EINVAL, "set_option: unknown option or bad value: " + n);
  }
  h->generation++;
  return B200MS_OK;
}

B200MS_API int64_t b200ms_corpus_pages(const b200ms_t* h) { return h ? h->corpus.n_pages : 0; }
B200MS_API int64_t b200ms_corpus_rows(const b200ms_t* h) { return h ? h->corpus.n_rows : 0; }

// ------------------------------------------------------------------------------------------------ quantise / pack
static int pack_items(b200ms_t* h, const void* src, int src_dtype, const int32_t* lens, int64_t n, bool queries,
                      void* dst, int dst_dtype, int64_t dst_rows_total, float i8_scale, cudaStream_t s,
                      std::vector<int64_t>* dst_start_out) {
  // one metadata block [ss | ds], one upload
  std::vector<int64_t> sd(2 * (size_t(n) + 1));
  int64_t* ss = sd.data();
  int64_t* ds = sd.data() + n + 1;
  ss[0] = ds[0] = 0;
  for (int64_t i = 0; i < n; ++i) {
    const int64_t len = lens[i] > 0 ? lens[i] : 0;
    ss[i + 1] = ss[i] + len;
    ds[i + 1] = ds[i] + b200ms_padded_len(len);
  }
  const int64_t dst_rows = dst_rows_total >= 0 ? dst_rows_total : ds[n];
  if (int e = upload(h, h->meta_b, sd.data(), sd.size() * 8, s)) return e;
  const int64_t* dev = static_cast<const int64_t*>(h->meta_b.p);
  if (int e = launch_pack_rows(h, src, src_dtype, dev, dev + n + 1, n, dst_rows, queries ? 1 : 0, dst, dst_dtype, i8_scale, s))
    return e;
  // sd is pageable host memory: cudaMemcpyAsync staged it before returning, so it may die here
  if (dst_start_out) dst_start_out->assign(ds, ds + n + 1);
  return B200MS_OK;
}

B200MS_API int b200ms_sign_pack(b200ms_t* h, const void* x, int src_dtype, int64_t rows, uint8_t* out, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype) || rows < 0 || (rows > 0 && (!x || !out)))
    return set_error(h, B200MS_EINVAL, "sign_pack: bad arguments");
  if (rows == 0) return B200MS_OK;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t st[2] = {0, rows};
  if (int e = upload(h, h->meta_b, st, sizeof(st), s)) return e;
  const int64_t* d = static_cast<const int64_t*>(h->meta_b.p);
  return launch_pack_rows(h, x, src_dtype, d, d, 1, rows, 0, out, B200MS_B1, 1.f, s);
}

B200MS_API int b200ms_hamming_batch(b200ms_t* h, const uint8_t* q_bits, const uint8_t* cand_bits, int64_t n, uint32_t* out,
                                    void* stream) {
  if (!h) return B200MS_EINVAL;
  if (n < 0 || (n > 0 && (!q_bits || !cand_bits || !out)) || (reinterpret_cast<uintptr_t>(q_bits) & 15) ||
      (reinterpret_cast<uintptr_t>(cand_bits) & 15))
    return set_error(h, B200MS_EINVAL, "hamming_batch: bad arguments (16-byte aligned packed rows)");
  DeviceGuard g(h->device);
  return launch_hamming_batch(h, q_bits, cand_bits, n, out, static_cast<cudaStream_t>(stream));
}

B200MS_API int b200ms_pack_pages(b200ms_t* h, const void* src, int src_dtype, const int32_t* page_lens, int64_t n_pages,
                                 void* dst, int dst_dtype, float i8_scale, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype) || !corpus_dtype_ok(dst_dtype) || n_pages < 0 || (n_pages > 0 && (!page_lens || !dst)))
    return set_error(h, B200MS_EINVAL, "pack_pages: bad arguments");
  if (n_pages == 0) return B200MS_OK;
  DeviceGuard g(h->device);
  return pack_items(h, src, src_dtype, page_lens, n_pages, false, dst, dst_dtype, -1, i8_scale,
                    static_cast<cudaStream_t>(stream), nullptr);
}

B200MS_API int b200ms_pack_queries(b200ms_t* h, const void* q, int src_dtype, const int32_t* q_lens, int n_q,
                                   void* q_packed, int dst_dtype, float i8_scale, int32_t* group_offsets_out,
                                   int* n_groups_out, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype) || !corpus_dtype_ok(dst_dtype) || n_q < 0 || (n_q > 0 && (!q_lens || !q_packed)))
    return set_error(h, B200MS_EINVAL, "pack_queries: bad arguments");
  DeviceGuard g(h->device);
  const int64_t groups = b200ms_query_groups(q_lens, n_q);
  const int64_t groups_padded = (groups + 3) & ~int64_t(3);
  std::vector<int64_t> ds;
  if (groups_padded > 0) {
    if (int e = pack_items(h, q, src_dtype, q_lens, n_q, true, q_packed, dst_dtype, groups_padded * kGroup, i8_scale,
                           static_cast<cudaStream_t>(stream), &ds))
      return e;
  } else {
    ds.assign(size_t(n_q) + 1, 0);
  }
  if (group_offsets_out)
    for (int i = 0; i <= n_q; ++i) group_offsets_out[i] = int32_t(ds[i] / kGroup);
  if (n_groups_out) *n_groups_out = int(groups);
  return B200MS_OK;
}

// ------------------------------------------------------------------------------------------------ corpus
B200MS_API int b200ms_set_corpus(b200ms_t* h, const void* rows, int dtype, const int32_t* page_lens, int64_t n_pages) {
  if (!h) return B200MS_EINVAL;
  if (!corpus_dtype_ok(dtype) || n_pages < 0 || (n_pages > 0 && (!rows || !page_lens)))
    return set_error(h, B200MS_EINVAL, "set_corpus: bad arguments");
  if (n_pages > 0 && (reinterpret_cast<uintptr_t>(rows) & 1023))
    return set_error(h, B200MS_EINVAL, "set_corpus: rows must be 1024-byte aligned");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  Corpus c;
  c.rows = rows;
  c.dtype = dtype;
  c.n_pages = n_pages;
  std::vector<int64_t> ps(size_t(n_pages) + 1);
  ps[0] = 0;
  for (int64_t i = 0; i < n_pages; ++i) {
    ps[i + 1] = ps[i] + b200ms_padded_len(page_lens[i]);
    if (page_lens[i] <= 0) c.has_empty = true;
  }
  c.n_rows = ps[n_pages];
  c.n_chunks = c.n_rows / kGroup;
  if (c.n_chunks >= (int64_t(1) << 31)) return set_error(h, B200MS_EINVAL, "set_corpus: more than 2^31 chunks");
  // work units: runs of whole pages of about unit_rows rows; unit_start in chunks
  // (small corpora: shrink the units so that every SM still gets about four of them -- a 100-page corpus as 25 units
  // of 4096 rows would leave 123 SMs idle)
  int64_t unit_rows = c.n_rows / (4 * int64_t(h->num_sms > 0 ? h->num_sms : 1));
  if (unit_rows < kTileN) unit_rows = kTileN;
  if (unit_rows > h->unit_rows) unit_rows = h->unit_rows;
  std::vector<int32_t> us;
  us.push_back(0);
  int64_t acc = 0;
  for (int64_t i = 0; i < n_pages; ++i) {
    acc += ps[i + 1] - ps[i];
    if (acc >= unit_rows) {
      us.push_back(int32_t(ps[i + 1] / kGroup));
      acc = 0;
    }
  }
  if (us.back() != int32_t(c.n_chunks)) us.push_back(int32_t(c.n_chunks));
  c.n_units = int(us.size()) - 1;
  if (int e = upload(h, h->page_start, ps.data(), ps.size() * 8, s)) return e;
  if (int e = upload(h, h->unit_start, us.data(), us.size() * 4, s)) return e;
  if (int e = upload(h, h->page_len, page_lens, size_t(n_pages) * 4, s)) return e;
  h->page_len_host.assign(page_lens, page_lens + n_pages);
  if (int e = reserve(h, h->chunk_page, size_t(c.n_chunks > 0 ? c.n_chunks : 1) * 4)) return e;
  if (int e = launch_chunk_page(h, static_cast<const int64_t*>(h->page_start.p), n_pages,
                                static_cast<int32_t*>(h->chunk_page.p), s))
    return e;
  if (dtype != B200MS_B1 && c.n_rows > 0) {
    if (int e = make_tmap_rows(h, &c.tmap, rows, dtype, c.n_rows, kTileN)) return e;
    c.has_tmap = true;
  }
  if (int e = check_cuda(h, cudaStreamSynchronize(s), "set_corpus: stream sync")) return e;
  h->corpus = c;
  h->generation++;
  return B200MS_OK;
}

// zero_pad_compat, full scan: pages are "batched" in page-id order, zero_pad_batch at a time (score_multi_vector's
// batch_size, 128 upstream); a page shorter than the longest of its batch gets its per-token maxima clamped at 0.
// Built on the host once per (corpus, batch size) and cached on the device.
static int ensure_clamp_pages(b200ms_t* h, cudaStream_t s, const uint32_t** out) {
  *out = nullptr;
  if (h->zero_pad_batch <= 0 || h->corpus.dtype == B200MS_B1) return B200MS_OK;  // SQL max_sim has no padding quirk
  Corpus& c = h->corpus;
  const int64_t n = c.n_pages;
  if (c.clamp_batch != h->zero_pad_batch) {
    std::vector<uint32_t> bits(size_t((n + 31) / 32) + 1, 0u);
    const int64_t B = h->zero_pad_batch;
    for (int64_t b0 = 0; b0 < n; b0 += B) {
      const int64_t b1 = b0 + B < n ? b0 + B : n;
      int32_t mx = 0;
      for (int64_t p = b0; p < b1; ++p) mx = h->page_len_host[p] > mx ? h->page_len_host[p] : mx;
      for (int64_t p = b0; p < b1; ++p)
        if (h->page_len_host[p] < mx) bits[size_t(p >> 5)] |= 1u << (p & 31);
    }
    if (int e = upload(h, h->clamp_pages, bits.data(), bits.size() * 4, s)) return e;
    c.clamp_batch = h->zero_pad_batch;
  }
  *out = static_cast<const uint32_t*>(h->clamp_pages.p);
  return B200MS_OK;
}

// ------------------------------------------------------------------------------------------------ hot path
// Candidate description for score_impl / search_impl.
//   ids == NULL           : scan the whole corpus, scores indexed by page id.
//   ids, per_query == 0   : ONE list of n_cand page ids (-1 = unused slot) scored by every query, scores indexed by slot.
//   ids, per_query == 1   : one list PER QUERY, ids = [n_q, stride] with stride = roundup(n_cand, 32); query q owns slots
//                           [q*stride, q*stride + n_cand) and only its own groups are scored against them.
struct CandSpec {
  const int64_t* ids = nullptr;
  int n_cand = 0;
  int per_query = 0;
  int64_t stride = 0;
  int64_t n_slots(int n_q) const { return per_query ? stride * n_q : n_cand; }
};

static int score_impl(b200ms_t* h, const void* q_packed, int n_groups, const int32_t* goff, int n_q, const int32_t* ntok_dev,
                      void* group_scores, int64_t ld, const CandSpec& cs, cudaStream_t s) {
  const Corpus& c = h->corpus;
  if (c.dtype < 0) return set_error(h, B200MS_ESTATE, "score: no corpus attached (call b200ms_set_corpus first)");
  const int64_t n_items = cs.ids ? cs.n_slots(n_q) : c.n_pages;
  if (n_groups < 0 || ld < n_items || cs.n_cand < 0 || (n_groups > 0 && (!q_packed || !group_scores)))
    return set_error(h, B200MS_EINVAL, "score: bad arguments");
  if (n_groups == 0 || n_items == 0 || c.n_pages == 0) return B200MS_OK;
  const int slot = int(h->ev_count % b200ms_t::kEvRing);
  const int n_groups_padded = (n_groups + 3) & ~3;
  if (c.dtype == B200MS_B1) {
    if (!goff || !ntok_dev || n_q <= 0) return set_error(h, B200MS_EINVAL, "score: B1 needs the per-group token counts");
    // b1_tensor: 0 = POPC kernel, 1 = tcgen05 kernel, 2 (default) = measured crossover: one 32-token group is faster on the
    // POPC pipe (1.59 vs 2.49 ms / 65536 pages), two or more groups on the tensor cores (a 128-token tile costs the same
    // as one token there).  Rerank of a candidate list stays on the POPC kernel.
    // A full scan of ONE group runs with the patch rows as the M operand and the expanded bits in TMEM (maxsim_rowm.cu).
    const bool rowm_path = !cs.ids && h->rowm && h->b1_tensor != 0 && n_groups == 1;
    const bool tensor_path = rowm_path || (!cs.ids && (h->b1_tensor == 1 || (h->b1_tensor == 2 && n_groups >= 2)));
    if ((tensor_path && c.has_empty) || cs.per_query)
      if (int e = check_cuda(h, cudaMemsetAsync(group_scores, 0, size_t(n_groups_padded) * size_t(ld) * 4, s), "score: memset")) return e;
    if (!h->capturing)
      if (int e = check_cuda(h, cudaEventRecord(h->ev0[slot], s), "score: event record")) return e;
    if (rowm_path) {
      if (int e = launch_score_rowm(h, q_packed, n_groups, ntok_dev, nullptr, group_scores, ld, s)) return e;
    } else if (tensor_path) {
      if (int e = launch_score_b1_umma(h, q_packed, ntok_dev, n_groups, group_scores, ld, s)) return e;
    } else if (cs.per_query) {
      for (int q = 0; q < n_q; ++q) {
        if (goff[q + 1] <= goff[q]) continue;
        if (int e = launch_score_b1(h, cs.ids + int64_t(q) * cs.stride, cs.n_cand, q_packed, n_groups, ntok_dev,
                                    static_cast<int32_t*>(group_scores) + int64_t(q) * cs.stride, ld, s, goff[q], goff[q + 1]))
          return e;
      }
    } else {
      if (int e = launch_score_b1(h, cs.ids, cs.n_cand, q_packed, n_groups, ntok_dev, group_scores, ld, s, 0, n_groups)) return e;
    }
    if (!h->capturing) {
      if (int e = check_cuda(h, cudaEventRecord(h->ev1[slot], s), "score: event record")) return e;
      h->ev_count++;
    }
    return B200MS_OK;
  }
  // pages with zero rows (and unused candidate slots) are never touched by the tile kernel: they score 0
  if (c.has_empty || cs.ids) {
    if (int e = check_cuda(h, cudaMemsetAsync(group_scores, 0, size_t(n_groups_padded) * size_t(ld) * 4, s), "score: memset")) return e;
  }
  UnitPlan plan;
  if (cs.ids) {
    const int n_slots = int(cs.n_slots(n_q));
    if (int e = reserve(h, h->cand_start, size_t(n_slots) * 4)) return e;
    if (int e = reserve(h, h->cand_end, size_t(n_slots) * 4)) return e;
    if (int e = launch_cand_units(h, cs.ids, n_slots, static_cast<int32_t*>(h->cand_start.p),
                                  static_cast<int32_t*>(h->cand_end.p), nullptr, s))
      return e;
    plan.start = static_cast<const int32_t*>(h->cand_start.p);
    plan.end = static_cast<const int32_t*>(h->cand_end.p);
    plan.n_units = n_slots;
    plan.slot_mode = 1;
    if (h->zero_pad_batch > 0) {  // the reference's quirk, exactly: batches of zero_pad_batch candidates in first-stage order
      if (int e = reserve(h, h->clamp_slots, size_t((n_slots + 31) / 32 + 1) * 4)) return e;
      const int lists = cs.per_query ? n_q : 1;
      const int64_t stride = cs.per_query ? cs.stride : 0;
      if (int e = launch_clamp_slots(h, cs.ids, cs.n_cand, lists, stride, h->zero_pad_batch,
                                     static_cast<uint32_t*>(h->clamp_slots.p), s))
        return e;
      plan.clamp_bits = static_cast<const uint32_t*>(h->clamp_slots.p);
    }
  } else {  // full scan: unit u = [unit_start[u], unit_start[u+1])
    plan.start = static_cast<const int32_t*>(h->unit_start.p);
    plan.end = plan.start + 1;
    plan.n_units = c.n_units;
    plan.slot_mode = 0;
    if (int e = ensure_clamp_pages(h, s, &plan.clamp_bits)) return e;
  }
  if (!h->capturing)
    if (int e = check_cuda(h, cudaEventRecord(h->ev0[slot], s), "score: event record")) return e;
  if (cs.ids && cs.per_query) {
    // one launch per 128-token query tile: the tile's queries against THEIR candidate lists only (a contiguous slot range)
    const int n_mtiles = n_groups_padded / 4;
    int q_lo = 0;
    for (int m = 0; m < n_mtiles; ++m) {
      const int g0 = 4 * m, g1 = 4 * m + 4;
      while (q_lo < n_q && goff[q_lo + 1] <= g0) ++q_lo;  // first query with a group in this tile
      int q_hi = q_lo;
      while (q_hi < n_q && goff[q_hi] < g1) ++q_hi;        // one past the last
      if (q_hi <= q_lo) continue;
      UnitPlan sub = plan;
      const int64_t s0 = int64_t(q_lo) * cs.stride;
      sub.start += s0;
      sub.end += s0;
      sub.n_units = int(int64_t(q_hi - q_lo) * cs.stride);
      if (sub.clamp_bits) sub.clamp_bits += s0 / 32;
      void* sc = static_cast<uint8_t*>(group_scores) + size_t(s0) * 4;
      if (int e = launch_score_umma(h, &sub, q_packed, n_groups, sc, ld, s, m)) return e;
    }
  } else if (!cs.ids && h->rowm && n_groups <= kRowmMaxGroups) {
    // the lone query: patch rows as the M operand, four epilogue warps in parallel (maxsim_rowm.cu)
    if (int e = launch_score_rowm(h, q_packed, n_groups, nullptr, plan.clamp_bits, group_scores, ld, s)) return e;
  } else {
    if (int e = launch_score_umma(h, &plan, q_packed, n_groups, group_scores, ld, s)) return e;
  }
  if (!h->capturing) {
    if (int e = check_cuda(h, cudaEventRecord(h->ev1[slot], s), "score: event record")) return e;
    h->ev_count++;
  }
  return B200MS_OK;
}

B200MS_API int b200ms_score(b200ms_t* h, const void* q_packed, int n_groups, const int32_t* q_lens,
                            const int32_t* group_offsets, int n_q, void* group_scores, int64_t ld, void* stream) {
  if (!h) return B200MS_EINVAL;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int32_t* ntok_dev = nullptr;
  if (h->corpus.dtype == B200MS_B1) {
    if (!q_lens || !group_offsets || n_q <= 0) return set_error(h, B200MS_EINVAL, "score: B1 needs q_lens and group_offsets");
    const int n_groups_padded = (n_groups + 3) & ~3;
    std::vector<int32_t> ntok(size_t(n_groups_padded > 0 ? n_groups_padded : 4), 0);
    for (int q = 0; q < n_q; ++q) {
      int left = q_lens[q];
      for (int gi = group_offsets[q]; gi < group_offsets[q + 1] && gi < n_groups; ++gi) {
        ntok[gi] = left > kGroup ? kGroup : left;
        left -= ntok[gi];
      }
    }
    if (int e = upload(h, h->meta, ntok.data(), ntok.size() * 4, s)) return e;
    ntok_dev = static_cast<const int32_t*>(h->meta.p);
  }
  return score_impl(h, q_packed, n_groups, group_offsets, n_q, ntok_dev, group_scores, ld, CandSpec{}, s);
}

static int score_time_of(b200ms_t* h, int64_t idx, float* ms) {
  const int slot = int(idx % b200ms_t::kEvRing);
  if (cudaEventSynchronize(h->ev1[slot]) != cudaSuccess) return check_cuda(h, cudaGetLastError(), "cudaEventSynchronize");
  if (cudaEventElapsedTime(ms, h->ev0[slot], h->ev1[slot]) != cudaSuccess) return check_cuda(h, cudaGetLastError(), "cudaEventElapsedTime");
  return B200MS_OK;
}

B200MS_API float b200ms_last_score_ms(b200ms_t* h) {
  if (!h) return float(B200MS_EINVAL);
  if (h->ev_count == 0) return float(set_error(h, B200MS_ESTATE, "last_score_ms: no scoring call recorded"));
  DeviceGuard g(h->device);
  float ms = 0.f;
  if (int e = score_time_of(h, h->ev_count - 1, &ms)) return float(e);
  return ms;
}

B200MS_API int64_t b200ms_score_call_count(const b200ms_t* h) { return h ? h->ev_count : 0; }

B200MS_API int b200ms_score_times_ms(b200ms_t* h, float* out_ms, int n) {
  if (!h || !out_ms || n < 0) return B200MS_EINVAL;
  if (n > b200ms_t::kEvRing || n > h->ev_count) return set_error(h, B200MS_EINVAL, "score_times_ms: n exceeds the recorded history (ring of 256)");
  DeviceGuard g(h->device);
  for (int i = 0; i < n; ++i)
    if (int e = score_time_of(h, h->ev_count - n + i, &out_ms[i])) return e;
  return n;
}

B200MS_API int b200ms_topk(b200ms_t* h, const void* group_scores, int score_dtype, int64_t n_pages, int64_t ld,
                           const int32_t* group_offsets, int n_q, const uint32_t* allow_mask, int k, float scale,
                           int64_t id_base, float* top_scores, int64_t* top_ids, int32_t* top_counts, void* stream) {
  if (!h) return B200MS_EINVAL;
  if ((score_dtype != B200MS_F32 && score_dtype != B200MS_I32) || n_pages < 0 || ld < n_pages || n_q < 0 || k < 1 ||
      k > B200MS_MAX_K || (n_q > 0 && (!group_offsets || !top_scores || !top_ids || !top_counts)) ||
      (n_q > 0 && n_pages > 0 && !group_scores))
    return set_error(h, B200MS_EINVAL, "topk: bad arguments (1 <= k <= 4096)");
  if (n_q == 0) return B200MS_OK;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int e = upload(h, h->meta, group_offsets, size_t(n_q + 1) * 4, s)) return e;
  return launch_topk(h, group_scores, score_dtype, n_pages, ld, static_cast<const int32_t*>(h->meta.p), n_q, allow_mask,
                     k, scale, id_base, nullptr, top_scores, top_ids, top_counts, s);
}

B200MS_API int b200ms_merge_topk(b200ms_t* h, const float* cand_scores, const int64_t* cand_ids, int n_q, int m, int k,
                                 float* top_scores, int64_t* top_ids, int32_t* top_counts, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (n_q < 0 || m < 1 || m > 2 * B200MS_MAX_K || k < 1 || k > B200MS_MAX_K ||
      (n_q > 0 && (!cand_scores || !cand_ids || !top_scores || !top_ids || !top_counts)))
    return set_error(h, B200MS_EINVAL, "merge_topk: bad arguments (m <= 8192, k <= 4096)");
  DeviceGuard g(h->device);
  return launch_merge_topk(h, cand_scores, cand_ids, n_q, m, k, top_scores, top_ids, top_counts,
                           static_cast<cudaStream_t>(stream));
}

namespace bms {

// The search step shared by every entry point: pack queries -> score -> top-k, all enqueued on `s`.
//   q_src           rows [sum q_lens,128] F32|BF16, device memory or (zero-copy path) mapped pinned host memory
//   meta_in_place   != NULL: the SearchMeta block already sits in device-readable memory at this address (mapped pinned
//                   staging) -- no upload; else the block is uploaded with ONE cudaMemcpyAsync
int search_core(b200ms_t* h, const void* q_src, int src_dtype, const int32_t* q_lens, int n_q, int k,
                const uint32_t* allow_dev, float i8_q_scale, float score_scale, int64_t id_base, float* ts, int64_t* ti,
                int32_t* tc, cudaStream_t s, const SearchCand* cand, const int32_t* mask_index_dev, int64_t mask_stride,
                const void* meta_in_place, const void* meta_host_block) {
  const Corpus& c = h->corpus;
  if (c.dtype < 0) return set_error(h, B200MS_ESTATE, "search: no corpus attached (call b200ms_set_corpus first)");
  if (n_q < 1 || !q_lens || !q_src || k < 1 || k > B200MS_MAX_K || !ts || !ti || !tc)
    return set_error(h, B200MS_EINVAL, "search: bad arguments (n_q >= 1, 1 <= k <= 4096)");
  SearchMeta local;
  const SearchMeta* m = static_cast<const SearchMeta*>(meta_host_block);
  if (!m) {
    build_search_meta(q_lens, n_q, &local);
    m = &local;
  }
  CandSpec cs;
  if (cand && cand->ids) {
    cs.ids = cand->ids;
    cs.n_cand = cand->n_cand;
    cs.per_query = cand->per_query;
    cs.stride = cand->per_query ? ((int64_t(cand->n_cand) + 31) & ~int64_t(31)) : 0;
    if (cs.per_query && cs.stride != cs.n_cand) {  // caller's lists are [n_q, n_cand]: give every list a 32-slot-aligned stride
      if (int e = reserve(h, h->cand_pad, size_t(cs.stride) * size_t(n_q) * 8)) return e;
      if (int e = launch_pad_cands(h, cand->ids, cs.n_cand, n_q, cs.stride, static_cast<int64_t*>(h->cand_pad.p), s)) return e;
      cs.ids = static_cast<const int64_t*>(h->cand_pad.p);
    }
  }
  const int64_t gp = m->groups_padded > 0 ? m->groups_padded : 4;
  const int64_t n_items = cs.ids ? cs.n_slots(n_q) : c.n_pages;
  const int64_t ld = ((n_items + 31) & ~int64_t(31)) > 0 ? ((n_items + 31) & ~int64_t(31)) : 32;
  if (int e = reserve(h, h->q_packed, size_t(gp) * kGroup * size_t(b200ms_row_bytes(c.dtype)))) return e;
  if (int e = reserve(h, h->scores, size_t(gp) * size_t(ld) * 4)) return e;
  const uint8_t* meta_dev = static_cast<const uint8_t*>(meta_in_place);
  if (!meta_dev) {
    if (int e = upload(h, h->meta, m->host.data(), m->host.size(), s)) return e;
    meta_dev = static_cast<const uint8_t*>(h->meta.p);
  }
  const int64_t* ss_dev = reinterpret_cast<const int64_t*>(meta_dev + m->off_ss);
  const int64_t* ds_dev = reinterpret_cast<const int64_t*>(meta_dev + m->off_ds);
  const int32_t* goff_dev = reinterpret_cast<const int32_t*>(meta_dev + m->off_goff);
  const int32_t* ntok_dev = reinterpret_cast<const int32_t*>(meta_dev + m->off_ntok);
  if (m->groups_padded > 0)
    if (int e = launch_pack_rows(h, q_src, src_dtype, ss_dev, ds_dev, n_q, m->groups_padded * kGroup, 1, h->q_packed.p, c.dtype,
                                 i8_q_scale, s))
      return e;
  const int ng = int(m->groups);
  if (int e = score_impl(h, h->q_packed.p, ng, m->goff.data(), n_q, ntok_dev, h->scores.p, ld, cs, s)) return e;
  if (ng == 0 || n_items == 0) {
    // nothing scored: every page (if any) has score 0 -- still a defined ranking
    if (int e = check_cuda(h, cudaMemsetAsync(h->scores.p, 0, size_t(gp) * size_t(ld) * 4, s), "search: memset")) return e;
  }
  const int sdt = (c.dtype == B200MS_BF16 || c.dtype == B200MS_F8) ? B200MS_F32 : B200MS_I32;
  if (!cs.ids) {
    return launch_topk(h, h->scores.p, sdt, c.n_pages, ld, goff_dev, n_q, allow_dev, k, score_scale, id_base, nullptr, ts, ti,
                       tc, s, mask_index_dev, mask_stride);
  }
  // candidate mode: rank the slots (ties -> lower slot = better first-stage rank), report the page ids; unused slots masked
  const int n_slots = int(cs.n_slots(n_q));
  if (int e = reserve(h, h->cand_mask, size_t((n_slots + 31) / 32 + 1) * 4)) return e;
  if (int e = launch_cand_units(h, cs.ids, n_slots, nullptr, nullptr, static_cast<uint32_t*>(h->cand_mask.p), s)) return e;
  return launch_topk(h, h->scores.p, sdt, cs.n_cand, ld, goff_dev, n_q, static_cast<const uint32_t*>(h->cand_mask.p), k,
                     score_scale, 0, cs.ids, ts, ti, tc, s, nullptr, 0, cs.per_query ? cs.stride : 0);
}

}  // namespace bms

static int search_impl(b200ms_t* h, const void* q_dev, int src_dtype, const int32_t* q_lens, int n_q, int k,
                       const uint32_t* allow_dev, float i8_q_scale, float score_scale, int64_t id_base, float* ts,
                       int64_t* ti, int32_t* tc, cudaStream_t s, const SearchCand* cand = nullptr,
                       const int32_t* mask_index_dev = nullptr, int64_t mask_stride = 0) {
  return search_core(h, q_dev, src_dtype, q_lens, n_q, k, allow_dev, i8_q_scale, score_scale, id_base, ts, ti, tc, s, cand,
                     mask_index_dev, mask_stride, nullptr, nullptr);
}

B200MS_API int b200ms_rerank_device(b200ms_t* h, const void* q_dev, int src_dtype, const int32_t* q_lens, int n_q,
                                    const int64_t* cand_ids_dev, int n_cand, int k, float i8_q_scale, float score_scale,
                                    float* top_scores_dev, int64_t* top_ids_dev, int32_t* top_counts_dev, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype) || !cand_ids_dev || n_cand < 1)
    return set_error(h, B200MS_EINVAL, "rerank_device: bad arguments (F32/BF16 queries, n_cand >= 1)");
  DeviceGuard g(h->device);
  SearchCand cand{cand_ids_dev, n_cand, 0};
  return search_impl(h, q_dev, src_dtype, q_lens, n_q, k, nullptr, i8_q_scale, score_scale, 0, top_scores_dev, top_ids_dev,
                     top_counts_dev, static_cast<cudaStream_t>(stream), &cand);
}

B200MS_API int b200ms_rerank_batch_device(b200ms_t* h, const void* q_dev, int src_dtype, const int32_t* q_lens, int n_q,
                                          const int64_t* cand_ids_dev, int n_cand, int k, float i8_q_scale, float score_scale,
                                          float* top_scores_dev, int64_t* top_ids_dev, int32_t* top_counts_dev, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype) || !cand_ids_dev || n_cand < 1 || n_q < 1 ||
      ((int64_t(n_cand) + 31) & ~int64_t(31)) * n_q >= (int64_t(1) << 30))
    return set_error(h, B200MS_EINVAL, "rerank_batch_device: bad arguments (F32/BF16 queries, n_cand >= 1, n_q*n_cand < 2^30)");
  DeviceGuard g(h->device);
  SearchCand cand{cand_ids_dev, n_cand, 1};
  return search_impl(h, q_dev, src_dtype, q_lens, n_q, k, nullptr, i8_q_scale, score_scale, 0, top_scores_dev, top_ids_dev,
                     top_counts_dev, static_cast<cudaStream_t>(stream), &cand);
}

B200MS_API int b200ms_search_device(b200ms_t* h, const void* q_dev, int src_dtype, const int32_t* q_lens, int n_q, int k,
                                    const uint32_t* allow_mask_dev, float i8_q_scale, float score_scale, int64_t id_base,
                                    float* top_scores_dev, int64_t* top_ids_dev, int32_t* top_counts_dev, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype)) return set_error(h, B200MS_EINVAL, "search_device: src dtype must be F32 or BF16");
  DeviceGuard g(h->device);
  return search_impl(h, q_dev, src_dtype, q_lens, n_q, k, allow_mask_dev, i8_q_scale, score_scale, id_base, top_scores_dev,
                     top_ids_dev, top_counts_dev, static_cast<cudaStream_t>(stream));
}

B200MS_API int b200ms_search_device_masked(b200ms_t* h, const void* q_dev, int src_dtype, const int32_t* q_lens, int n_q,
                                           int k, const uint32_t* allow_masks_dev, int n_masks,
                                           const int32_t* mask_index_dev, float i8_q_scale, float score_scale,
                                           int64_t id_base, float* top_scores_dev, int64_t* top_ids_dev,
                                           int32_t* top_counts_dev, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (!src_dtype_ok(src_dtype)) return set_error(h, B200MS_EINVAL, "search_device_masked: src dtype must be F32 or BF16");
  if (n_masks < 0 || (n_masks > 0 && (!allow_masks_dev || !mask_index_dev)))
    return set_error(h, B200MS_EINVAL, "search_device_masked: n_masks > 0 needs the mask matrix and one index per query");
  DeviceGuard g(h->device);
  return search_impl(h, q_dev, src_dtype, q_lens, n_q, k, n_masks > 0 ? allow_masks_dev : nullptr, i8_q_scale, score_scale,
                     id_base, top_scores_dev, top_ids_dev, top_counts_dev, static_cast<cudaStream_t>(stream), nullptr,
                     n_masks > 0 ? mask_index_dev : nullptr, (h->corpus.n_pages + 31) / 32);
}

// Host entry point.  Two transports, same kernels:
//   zero-copy (small calls, the interactive case: <= 256 query rows and <= 64 KB of results): the query rows and the
//     per-call metadata are written into ONE handle-owned mapped pinned block that the pack / top-k kernels read in
//     place, and the top-k kernel writes its results straight into the same block -- no copy-engine operation and no
//     metadata upload on the critical path (round 1 spent ~12 driver calls, 4 of them pageable uploads, around a 15 us scan).
//   copy engine (batches): one H2D of the rows, one upload of the metadata block, one fused D2H of [scores|ids|counts].
static int search_host_impl(b200ms_t* h, const float* q_host, const int32_t* q_lens, int n_q, int k,
                            const uint32_t* masks_host, int n_masks, const int32_t* mask_index_host, float i8_q_scale,
                            float score_scale, int64_t id_base, float* top_scores_host, int64_t* top_ids_host,
                            int32_t* top_counts_host) {
  if (n_q < 1 || !q_lens || !q_host || k < 1 || k > B200MS_MAX_K || !top_scores_host || !top_ids_host || !top_counts_host)
    return set_error(h, B200MS_EINVAL, "search_host: bad arguments (n_q >= 1, 1 <= k <= 4096)");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  SearchMeta m;
  build_search_meta(q_lens, n_q, &m);
  const size_t q_bytes = size_t(m.rows > 0 ? m.rows : 0) * kDim * 4;
  const size_t nk = size_t(n_q) * size_t(k);
  const size_t out_ids_off = 0, out_scores_off = nk * 8, out_counts_off = nk * 12;
  const size_t out_bytes = (nk * 12 + size_t(n_q) * 4 + 15) & ~size_t(15);
  const uint32_t* allow_dev = nullptr;
  const int32_t* index_dev = nullptr;
  const int64_t words = (h->corpus.n_pages + 31) / 32;
  if (masks_host && n_masks > 0 && h->corpus.n_pages > 0) {
    if (mask_index_host)
      for (int i = 0; i < n_q; ++i)
        if (mask_index_host[i] < -1 || mask_index_host[i] >= n_masks)
          return set_error(h, B200MS_EINVAL, "search_host_masked: mask_index out of range");
    if (int e = upload(h, h->mask, masks_host, size_t(n_masks) * size_t(words) * 4, s)) return e;
    allow_dev = static_cast<const uint32_t*>(h->mask.p);
    if (mask_index_host) {
      if (int e = upload(h, h->mask_index, mask_index_host, size_t(n_q) * 4, s)) return e;
      index_dev = static_cast<const int32_t*>(h->mask_index.p);
    }
  }
  const bool zc = h->zero_copy && m.rows <= 256 && out_bytes <= (64u << 10);
  const size_t meta_off = 0, q_off = (m.host.size() + 255) & ~size_t(255), out_off = (q_off + q_bytes + 255) & ~size_t(255);
  if (int e = reserve_pinned(h, h->stage, out_off + out_bytes)) return e;
  uint8_t* st = static_cast<uint8_t*>(h->stage.p);
  int e = 0;
  if (zc) {
    memcpy(st + meta_off, m.host.data(), m.host.size());
    if (q_bytes) memcpy(st + q_off, q_host, q_bytes);
    float* ts = reinterpret_cast<float*>(st + out_off + out_scores_off);
    int64_t* ti = reinterpret_cast<int64_t*>(st + out_off + out_ids_off);
    int32_t* tc = reinterpret_cast<int32_t*>(st + out_off + out_counts_off);
    // Small unmasked calls repeat with the same shapes (interactive queries): the second call of a shape is captured into
    // a CUDA graph -- pack -> score -> top-k become ONE launch, the third call onwards replays it.  Everything the kernels
    // read or write sits at fixed addresses (mapped staging block, handle scratch); h->generation changes when any moves.
    b200ms::HostGraph* hg = nullptr;  // NOLINT
    if (h->host_graph && !allow_dev) {
      uint64_t key = 1469598103934665603ull;
      auto mix = [&](uint64_t v) { key = (key ^ v) * 1099511628211ull; };
      mix(uint64_t(n_q));
      mix(uint64_t(k));
      for (int i = 0; i < n_q; ++i) mix(uint64_t(uint32_t(q_lens[i])));
      mix(uint64_t(id_base));
      uint32_t fb;
      memcpy(&fb, &score_scale, 4);
      mix(fb);
      memcpy(&fb, &i8_q_scale, 4);
      mix(fb);
      for (auto& g2 : h->host_graphs)
        if (g2.key == key) hg = &g2;
      if (!hg) {
        if (h->host_graphs.size() >= 16) {  // evict the least recently used shape
          size_t lru = 0;
          for (size_t i = 1; i < h->host_graphs.size(); ++i)
            if (h->host_graphs[i].last_use < h->host_graphs[lru].last_use) lru = i;
          if (h->host_graphs[lru].exec) cudaGraphExecDestroy(h->host_graphs[lru].exec);
          h->host_graphs.erase(h->host_graphs.begin() + long(lru));
        }
        h->host_graphs.emplace_back();
        hg = &h->host_graphs.back();
        hg->key = key;
      }
      hg->last_use = ++h->graph_clock;
      if (hg->exec && hg->generation != h->generation) {  // a buffer moved / corpus or option changed: start over
        cudaGraphExecDestroy(hg->exec);
        hg->exec = nullptr;
        hg->seen = 0;
      }
    }
    if (hg && hg->exec) {
      if (int e2 = check_cuda(h, cudaGraphLaunch(hg->exec, s), "search_host: graph launch")) return e2;
      h->launches += hg->launches;
    } else if (hg && hg->seen >= 1) {
      const uint64_t gen0 = h->generation;
      const int64_t l0 = h->launches;
      if (int e2 = check_cuda(h, cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal), "search_host: begin capture")) return e2;
      h->capturing = true;
      e = search_core(h, st + q_off, B200MS_F32, q_lens, n_q, k, nullptr, i8_q_scale, score_scale, id_base, ts, ti, tc, s, nullptr,
                      nullptr, words, st + meta_off, &m);
      h->capturing = false;
      cudaGraph_t graph = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(s, &graph);
      if (e || ce != cudaSuccess || !graph || gen0 != h->generation) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        hg->seen = -1000000;  // this shape does not capture: plain launches from now on
        e = search_core(h, st + q_off, B200MS_F32, q_lens, n_q, k, nullptr, i8_q_scale, score_scale, id_base, ts, ti, tc, s,
                        nullptr, nullptr, words, st + meta_off, &m);
        if (e) return e;
      } else {
        const cudaError_t ie = cudaGraphInstantiate(&hg->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) {
          cudaGetLastError();
          hg->exec = nullptr;
          hg->seen = -1000000;
          e = search_core(h, st + q_off, B200MS_F32, q_lens, n_q, k, nullptr, i8_q_scale, score_scale, id_base, ts, ti, tc, s,
                          nullptr, nullptr, words, st + meta_off, &m);
          if (e) return e;
        } else {
          hg->generation = h->generation;
          hg->launches = int(h->launches - l0);
          if (int e2 = check_cuda(h, cudaGraphLaunch(hg->exec, s), "search_host: graph launch")) return e2;
        }
      }
    } else {
      if (hg) hg->seen++;
      e = search_core(h, st + q_off, B200MS_F32, q_lens, n_q, k, allow_dev, i8_q_scale, score_scale, id_base, ts, ti, tc, s,
                      nullptr, index_dev, words, st + meta_off, &m);
      if (e) return e;
    }
  } else {
    if (int e2 = reserve(h, h->q_raw, q_bytes ? q_bytes : 512)) return e2;
    if (int e2 = reserve(h, h->out_all, out_bytes)) return e2;
    if (q_bytes)
      if (int e2 = check_cuda(h, cudaMemcpyAsync(h->q_raw.p, q_host, q_bytes, cudaMemcpyHostToDevice, s), "search_host: H2D queries")) return e2;
    uint8_t* od = static_cast<uint8_t*>(h->out_all.p);
    e = search_core(h, h->q_raw.p, B200MS_F32, q_lens, n_q, k, allow_dev, i8_q_scale, score_scale, id_base,
                    reinterpret_cast<float*>(od + out_scores_off), reinterpret_cast<int64_t*>(od + out_ids_off),
                    reinterpret_cast<int32_t*>(od + out_counts_off), s, nullptr, index_dev, words, nullptr, &m);
    if (e) return e;
    if (int e2 = check_cuda(h, cudaMemcpyAsync(st + out_off, od, out_bytes, cudaMemcpyDeviceToHost, s), "search_host: D2H results")) return e2;
  }
  if (int e2 = check_cuda(h, cudaStreamSynchronize(s), "search_host: stream sync")) return e2;
  memcpy(top_ids_host, st + out_off + out_ids_off, nk * 8);
  memcpy(top_scores_host, st + out_off + out_scores_off, nk * 4);
  memcpy(top_counts_host, st + out_off + out_counts_off, size_t(n_q) * 4);
  return B200MS_OK;
}

B200MS_API int b200ms_search_host(b200ms_t* h, const float* q_host, const int32_t* q_lens, int n_q, int k,
                                  const uint32_t* allow_mask_host, float i8_q_scale, float score_scale, int64_t id_base,
                                  float* top_scores_host, int64_t* top_ids_host, int32_t* top_counts_host) {
  if (!h) return B200MS_EINVAL;
  return search_host_impl(h, q_host, q_lens, n_q, k, allow_mask_host, allow_mask_host ? 1 : 0, nullptr, i8_q_scale,
                          score_scale, id_base, top_scores_host, top_ids_host, top_counts_host);
}

B200MS_API int b200ms_search_host_masked(b200ms_t* h, const float* q_host, const int32_t* q_lens, int n_q, int k,
                                         const uint32_t* allow_masks_host, int n_masks, const int32_t* mask_index_host,
                                         float i8_q_scale, float score_scale, int64_t id_base, float* top_scores_host,
                                         int64_t* top_ids_host, int32_t* top_counts_host) {
  if (!h) return B200MS_EINVAL;
  if (n_masks < 0 || (n_masks > 0 && (!allow_masks_host || !mask_index_host)))
    return set_error(h, B200MS_EINVAL, "search_host_masked: n_masks > 0 needs the mask matrix and one index per query");
  return search_host_impl(h, q_host, q_lens, n_q, k, allow_masks_host, n_masks, mask_index_host, i8_q_scale, score_scale,
                          id_base, top_scores_host, top_ids_host, top_counts_host);
}
