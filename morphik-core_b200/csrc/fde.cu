// fde.cu -- fixed-dimensional encodings (MUVERA FDE) and the dense candidate scan over them.
//
// Replaces stage 1-2 of FastMultiVectorStore.query_similar (core/vector_store/fast_multivector_store.py:521-532):
//   fde.generate_query_encoding / generate_document_encoding (C++ extension `fixed_dimensional_encoding`, configured at
//   :325-331 with dimension=128, num_repetitions=20, num_simhash_projections=5, projection_dimension=16, AMS_SKETCH)
//   + the Turbopuffer ANN query with distance_metric="cosine_distance" (:497,:526-532)
// by an exact device-side encoder and an exhaustive cosine scan of the [N, 10240] FDE matrix.
// The extension's sources are NOT in the reference snapshot (fde/ ships only pyproject.toml, SURVEY F2): the algorithm
// below restates the published MUVERA construction; the random matrices come from the host (fde.py, or a caller who has
// the upstream ones) -- parity with the upstream RNG stream is unpinned and documented as such.
//
// Per repetition r:  partition(x) = gray-code index of the sign bits of x * G_r (G_r: [128, ksim] Gaussian),
//                    proj(x)[j]  = scale * sum_{i : idx_r[i] == j} sign_r[i] * x[i]        (AMS / count sketch, 128 -> proj)
//                    block[r][partition] += proj(x)      (queries: SUM;  documents: SUM / count = AVERAGE, empty -> 0, or
//                    with fill_empty_partitions the projection of the point whose sign bits are nearest in Hamming distance)
// Optional final projection (final_projection_dimension): a count sketch of the whole vector, out[j] = sum sign_i * v_i.
// Deterministic: no atomics -- thread (partition, j) walks the rows in order, so the result is bit-identical to the
// oracle's loops (oracle/fde_oracle.c) in fp32.
//
// Scan: scores[q, p] = <q_fde[q], F[p]> * inv_norm[p].  HBM-bound (2 * fde_dim bytes per page, 20 KB in the reference
// configuration) -- fde_scan_umma_kernel streams the matrix ONCE per batch of up to 128 queries through tcgen05
// (pages = M, queries = N), fde_scan_kernel is the SIMT fallback for shapes the tensor path does not take.
#include <cuda_bf16.h>

#include "common.cuh"
#include "ptx.cuh"
#include "umma_tile.cuh"

namespace bms {

constexpr int kFdeMaxSeg = 2048;  // rows whose partition ids are staged in shared memory at a time
constexpr int kFdeThreads = 512;  // = 32 partitions x 16 projection dims for the reference configuration

__device__ __forceinline__ float load_elem(const void* src, int src_dtype, int64_t row, int d) {
  if (src_dtype == B200MS_F32) return __ldg(static_cast<const float*>(src) + row * kDim + d);
  const uint16_t raw = __ldg(static_cast<const uint16_t*>(src) + row * kDim + d);
  return __uint_as_float(uint32_t(raw) << 16);
}

// grid = (n_items, reps); block = kFdeThreads
__global__ void __launch_bounds__(kFdeThreads)
fde_encode_kernel(const void* __restrict__ rows, int src_dtype, const int64_t* __restrict__ item_start,
                  const int32_t* __restrict__ item_len /* NULL: items are back to back (item_start[i+1] ends item i) */,
                  const float* __restrict__ simhash /*[reps,128,ksim]*/, const int32_t* __restrict__ ams_index /*[reps,128]*/,
                  const float* __restrict__ ams_sign /*[reps,128]*/, int ksim, int proj, float scale, int is_document,
                  int fill_empty, float* __restrict__ out /*[n_items, reps * 2^ksim * proj]*/) {
  __shared__ float s_g[kDim * 8];          // G_r, [128][ksim] (ksim <= 8)
  __shared__ int s_off[65];                // CSR of the AMS sketch: dims of bucket j are s_dims[s_off[j] .. s_off[j+1])
  __shared__ uint8_t s_dims[kDim];
  __shared__ float s_sgn[kDim];
  __shared__ uint8_t s_part[kFdeMaxSeg];
  const int item = blockIdx.x, rep = blockIdx.y, reps = gridDim.y;
  const int n_part = 1 << ksim;
  const int tid = threadIdx.x;
  for (int i = tid; i < kDim * ksim; i += blockDim.x) s_g[i] = simhash[int64_t(rep) * kDim * ksim + i];
  if (tid == 0) {  // counting sort of the 128 input dims by bucket (ascending dim inside a bucket)
    int cnt[64];
    for (int j = 0; j < proj; ++j) cnt[j] = 0;
    for (int i = 0; i < kDim; ++i) cnt[ams_index[rep * kDim + i]]++;
    int acc = 0;
    for (int j = 0; j < proj; ++j) {
      s_off[j] = acc;
      acc += cnt[j];
      cnt[j] = s_off[j];
    }
    s_off[proj] = acc;
    for (int i = 0; i < kDim; ++i) {
      const int j = ams_index[rep * kDim + i];
      s_dims[cnt[j]] = uint8_t(i);
      s_sgn[cnt[j]] = ams_sign[rep * kDim + i];
      cnt[j]++;
    }
  }
  __syncthreads();
  const int64_t r0 = item_start[item], r1 = item_len ? r0 + max(item_len[item], 0) : item_start[item + 1];
  const int my_part = tid / proj, my_j = tid % proj;
  const bool worker = my_part < n_part;
  // raw sign bits of a Gray-code index g: g ^ (g >> 1)   (inverse of the append rule idx = (idx << 1) + (bit ^ (idx & 1)))
  const uint32_t my_bits = uint32_t(my_part) ^ (uint32_t(my_part) >> 1);
  float acc = 0.f;
  int count = 0;
  int best_dist = 1 << 20;  // fill_empty_partitions: nearest point (Hamming distance of sign bits; first minimum wins)
  int64_t best_row = -1;
  for (int64_t seg = r0; seg < r1; seg += kFdeMaxSeg) {
    const int n = int(r1 - seg < kFdeMaxSeg ? r1 - seg : kFdeMaxSeg);
    // phase 1: SimHash partition of every row of the segment (one thread per row)
    for (int r = tid; r < n; r += blockDim.x) {
      float dot[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) dot[k] = 0.f;
      for (int d = 0; d < kDim; ++d) {
        const float x = load_elem(rows, src_dtype, seg + r, d);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < ksim) dot[k] = fmaf(x, s_g[d * ksim + k], dot[k]);
      }
      uint32_t code = 0;  // Gray-code append: idx = (idx << 1) + (bit ^ (idx & 1))
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < ksim) code = (code << 1) + (uint32_t(dot[k] > 0.f) ^ (code & 1u));
      s_part[r] = uint8_t(code);
    }
    __syncthreads();
    // phase 2: thread (partition, j) accumulates bucket j of the rows that fell into its partition, in row order
    if (worker) {
      const int e0 = s_off[my_j], e1 = s_off[my_j + 1];
      for (int r = 0; r < n; ++r) {
        const uint32_t code = s_part[r];
        if (code != uint32_t(my_part)) {
          if (fill_empty && count == 0) {
            const int dist = __popc((code ^ (code >> 1)) ^ my_bits);
            if (dist < best_dist) {
              best_dist = dist;
              best_row = seg + r;
            }
          }
          continue;
        }
        count++;
        float v = 0.f;
        for (int e = e0; e < e1; ++e) v += s_sgn[e] * load_elem(rows, src_dtype, seg + r, s_dims[e]);
        acc += v;
      }
    }
    __syncthreads();
  }
  if (worker) {
    float v = acc * scale;
    if (is_document) {
      if (count > 0) {
        v = v / float(count);
      } else if (fill_empty && best_row >= 0) {
        float w = 0.f;
        for (int e = s_off[my_j]; e < s_off[my_j + 1]; ++e) w += s_sgn[e] * load_elem(rows, src_dtype, best_row, s_dims[e]);
        v = w * scale;
      } else {
        v = 0.f;
      }
    }
    out[(int64_t(item) * reps + rep) * n_part * proj + my_part * proj + my_j] = v;
  }
}

// Final count-sketch projection: out[item, j] = sum over i in bucket j (ascending i) of sign[i] * v[item, i].
// CSR (off [final_dim+1], dims / signs permuted by bucket) is built on the host at configure time.
__global__ void __launch_bounds__(256)
fde_final_project_kernel(const float* __restrict__ v, int64_t n_items, int inner_dim, int final_dim,
                         const int32_t* __restrict__ csr /*[final_dim+1 offsets | inner_dim dims]*/,
                         const float* __restrict__ sgn /*[inner_dim], permuted*/, float* __restrict__ out) {
  const int64_t total = n_items * final_dim;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int64_t item = t / final_dim;
    const int j = int(t % final_dim);
    const int e0 = __ldg(csr + j), e1 = __ldg(csr + j + 1);
    const int32_t* dims = csr + final_dim + 1;
    float acc = 0.f;
    for (int e = e0; e < e1; ++e) acc += __ldg(sgn + e) * __ldg(v + item * inner_dim + __ldg(dims + e));
    out[t] = acc;
  }
}

// fp32 FDE rows -> bf16 rows of the FDE corpus + 1/||row|| (of the bf16-rounded row; 0 for an all-zero row)
__global__ void __launch_bounds__(256)
fde_finalize_kernel(const float* __restrict__ fde, int64_t n, int fde_dim, __nv_bfloat16* __restrict__ out_rows,
                    float* __restrict__ inv_norm) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t warp_stride = (int64_t(gridDim.x) * blockDim.x) >> 5;
  for (int64_t r = warp_global; r < n; r += warp_stride) {
    float ss = 0.f;
    for (int d = lane; d < fde_dim; d += 32) {
      const __nv_bfloat16 b = __float2bfloat16_rn(fde[r * fde_dim + d]);
      out_rows[r * fde_dim + d] = b;
      const float f = __bfloat162float(b);
      ss = fmaf(f, f, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) inv_norm[r] = ss > 0.f ? rsqrtf(ss) : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------ SIMT scan (fallback)
// One warp per page row, 16-byte loads, up to kFdeQ queries resident in shared memory.
constexpr int kFdeQ = 4;
__global__ void __launch_bounds__(256)
fde_scan_kernel(const uint4* __restrict__ F, const float* __restrict__ inv_norm, int64_t n_pages, int fde_dim,
                const float* __restrict__ q_fde, int n_q, int q_base, float* __restrict__ scores, int64_t ld) {
  extern __shared__ float s_q[];  // [nq_here][fde_dim]
  const int nq_here = min(kFdeQ, n_q - q_base);
  for (int i = threadIdx.x; i < nq_here * fde_dim; i += blockDim.x) s_q[i] = q_fde[int64_t(q_base) * fde_dim + i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t warp_stride = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int vec_per_row = fde_dim / 8;  // uint4 = 8 bf16
  for (int64_t p = warp_global; p < n_pages; p += warp_stride) {
    float acc[kFdeQ];
#pragma unroll
    for (int q = 0; q < kFdeQ; ++q) acc[q] = 0.f;
    const uint4* row = F + p * vec_per_row;
    // 4 independent 16-byte loads in flight per lane (the scan is latency-bound otherwise: one warp per 20 KB row)
    for (int v0 = lane; v0 < vec_per_row; v0 += 128) {
      uint4 w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int v = v0 + 32 * u;
        w[u] = v < vec_per_row ? __ldg(row + v) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int v = v0 + 32 * u;
        if (v >= vec_per_row) break;
        float f[8];
        f[0] = __uint_as_float(w[u].x << 16); f[1] = __uint_as_float(w[u].x & 0xffff0000u);
        f[2] = __uint_as_float(w[u].y << 16); f[3] = __uint_as_float(w[u].y & 0xffff0000u);
        f[4] = __uint_as_float(w[u].z << 16); f[5] = __uint_as_float(w[u].z & 0xffff0000u);
        f[6] = __uint_as_float(w[u].w << 16); f[7] = __uint_as_float(w[u].w & 0xffff0000u);
#pragma unroll
        for (int q = 0; q < kFdeQ; ++q) {
          if (q < nq_here) {
            const float4* qq = reinterpret_cast<const float4*>(s_q + q * fde_dim + v * 8);
            const float4 q0 = qq[0], q1 = qq[1];
            acc[q] = fmaf(f[0], q0.x, acc[q]); acc[q] = fmaf(f[1], q0.y, acc[q]);
            acc[q] = fmaf(f[2], q0.z, acc[q]); acc[q] = fmaf(f[3], q0.w, acc[q]);
            acc[q] = fmaf(f[4], q1.x, acc[q]); acc[q] = fmaf(f[5], q1.y, acc[q]);
            acc[q] = fmaf(f[6], q1.z, acc[q]); acc[q] = fmaf(f[7], q1.w, acc[q]);
          }
        }
      }
    }
    const float inv = __ldg(inv_norm + p);
#pragma unroll
    for (int q = 0; q < kFdeQ; ++q) {
      if (q < nq_here) {
        const float s = warp_sum(acc[q]);
        if (lane == 0) scores[int64_t(q_base + q) * ld + p] = s * inv;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ tcgen05 scan
// D[128 pages x NQP] = F_tile[128 x fde_dim] * Qb[NQP x fde_dim]^T on the tensor cores, fp32 accumulation in TMEM.
//   A (M side) = 128 consecutive FDE rows, streamed from HBM by TMA in K-blocks of 64 bf16 (16 KB, SWIZZLE_128B);
//   B (N side) = the query FDEs as bf16 rows: row q = hi(q_fde[q]) and row H+q = lo = bf16(q_fde[q] - hi), so that
//                D[:, q] + D[:, H+q] reproduces the fp32 query to ~2^-17 relative (the FDE corpus itself is bf16);
//                re-read per K-block from L2 (NQP * 128 B beside the 16 KB of A; evict_last keeps it resident).
// The matrix is read ONCE for up to 128 queries; one query costs the same HBM pass (it is the bandwidth that is paid for).
// Persistent, one CTA per SM, 256 threads: warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7
// epilogue (thread = one page of the tile: adds the hi/lo halves, scales by 1/||F_p||, writes scores[q, p] -- for a fixed
// q the 32 lanes of a warp write 32 consecutive pages, one coalesced 128-byte store).
// Algorithmic bytes per page: 2 * fde_dim (+ 4 * n_q of scores written).
constexpr int kScanThreads = 256;
constexpr uint32_t kScanATile = 128 * 128;  // 128 rows x 64 bf16

__global__ void __launch_bounds__(kScanThreads, 1)
fde_scan_umma_kernel(const __grid_constant__ CUtensorMap tmap_f, const __grid_constant__ CUtensorMap tmap_q,
                     const float* __restrict__ inv_norm, int64_t n_pages, int n_kblocks, int n_q, int q_base, int half_cols,
                     float* __restrict__ scores, int64_t ld, int num_stages) {
  const int nqp = 2 * half_cols;                        // MMA N: hi rows [0, H), lo rows [H, 2H)
  const uint32_t b_bytes = uint32_t(nqp) * 128u;
  const uint32_t stage_bytes = kScanATile + b_bytes;    // multiples of 1024 (nqp % 32 == 0)
  extern __shared__ uint8_t smem_raw[];
  const TileSmem sm = carve_tile_smem(smem_raw, 0, stage_bytes, num_stages);  // stage = A tile | B (queries)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t n_tiles = (n_pages + 127) / 128;
  // two accumulators; tempty: one arrive per epilogue warp
  const uint32_t tmem_base = tile_prologue<false>(sm, warp, &tmap_f, &tmap_q, num_stages, 1, 2, 4);

  if (warp == 0) {
    if (lane == 0) {
      const uint64_t pol_f = policy_evict_first();
      const uint64_t pol_q = policy_evict_last();
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int kb = 0; kb < n_kblocks; ++kb) {
          mbar_wait(&sm.empty[stage], phase ^ 1);
          mbar_expect_tx(&sm.full[stage], stage_bytes);
          uint8_t* a = sm.st + size_t(stage) * stage_bytes;
          tma_load_2d(&tmap_f, &sm.full[stage], a, kb * 64, int32_t(tile * 128), pol_f);
          tma_load_2d(&tmap_q, &sm.full[stage], a + kScanATile, kb * 64, 0, pol_q);
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = umma_idesc(0, 128, nqp);
    int stage = 0;
    uint32_t phase = 0;
    uint32_t t = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t buf = t & 1;
      mbar_wait(&sm.tempty[buf], ((t >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * 256;
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait(&sm.full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = smem_u32(sm.st + size_t(stage) * stage_bytes);
          const uint64_t ad = umma_desc_kmajor_sw128(a_addr);
          const uint64_t bd = umma_desc_kmajor_sw128(a_addr + kScanATile);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) umma_ss<0>(d_tmem, ad + ks * 2, bd + ks * 2, idesc, (kb | ks) != 0);
          umma_commit(&sm.empty[stage]);
          if (kb == n_kblocks - 1) umma_commit(&sm.tfull[buf]);
        }
        __syncwarp();
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    const int quad = warp & 3;
    const uint32_t lane_base = tmem_base + (uint32_t(quad * 32) << 16);
    uint32_t t = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t buf = t & 1;
      const int64_t p = tile * 128 + quad * 32 + lane;
      const float inv = p < n_pages ? __ldg(inv_norm + p) : 0.f;
      mbar_wait(&sm.tfull[buf], (t >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = lane_base + buf * 256;
      if (half_cols == 16) {  // <= 16 queries: hi and lo halves sit in one 32-column load
        uint32_t v[32];
        tmem_ld_32x32(taddr, v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.tempty[buf]);
        if (p < n_pages) {
#pragma unroll
          for (int q = 0; q < 16; ++q)
            if (q < n_q) scores[int64_t(q_base + q) * ld + p] = (__uint_as_float(v[q]) + __uint_as_float(v[16 + q])) * inv;
        }
      } else {
        for (int c = 0; c < half_cols; c += 32) {
          uint32_t hi[32], lo[32];
          tmem_ld_32x32(taddr + c, hi);
          tmem_ld_32x32(taddr + half_cols + c, lo);
          tmem_ld_wait();
          if (c + 32 >= half_cols) {  // last chunk read: the accumulator may be overwritten
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.tempty[buf]);
          }
          if (p < n_pages) {
#pragma unroll
            for (int q = 0; q < 32; ++q)
              if (c + q < n_q) scores[int64_t(q_base + c + q) * ld + p] = (__uint_as_float(hi[q]) + __uint_as_float(lo[q])) * inv;
          }
        }
      }
    }
  }
  tile_teardown<false>(warp, tmem_base);
}

// q_fde fp32 [n_q, fde_dim] (queries q_base ..) -> bf16 [2*half_cols, fde_dim]: rows [0,n) hi, rows [H, H+n) lo, rest zero
__global__ void __launch_bounds__(256)
fde_q_split_kernel(const float* __restrict__ q_fde, int n_here, int fde_dim, int half_cols, __nv_bfloat16* __restrict__ out) {
  const int64_t total = int64_t(2 * half_cols) * fde_dim;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int row = int(t / fde_dim), d = int(t % fde_dim);
    const int q = row < half_cols ? row : row - half_cols;
    float v = 0.f;
    if (q < n_here) {
      const float x = __ldg(q_fde + int64_t(q) * fde_dim + d);
      const float hi = __bfloat162float(__float2bfloat16_rn(x));
      v = row < half_cols ? hi : x - hi;
    }
    out[t] = __float2bfloat16_rn(v);
  }
}

int launch_fde_encode(b200ms_t* h, const void* rows, int src_dtype, const int64_t* item_start_dev, int n_items,
                      int is_document, float* out, cudaStream_t s, const int32_t* item_len_dev) {
  if (n_items <= 0) return B200MS_OK;
  dim3 grid(n_items, h->fde_reps);
  fde_encode_kernel<<<grid, kFdeThreads, 0, s>>>(rows, src_dtype, item_start_dev, item_len_dev,
                                                static_cast<const float*>(h->fde_simhash.p),
                                                static_cast<const int32_t*>(h->fde_ams_index.p),
                                                static_cast<const float*>(h->fde_ams_sign.p), h->fde_ksim, h->fde_proj,
                                                h->fde_scale, is_document, h->fde_fill_empty, out);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "launch fde_encode");
}

int launch_fde_finalize(b200ms_t* h, const float* fde, int64_t n, void* out_rows, float* inv_norm, cudaStream_t s) {
  if (n <= 0) return B200MS_OK;
  int64_t blocks = (n + 7) / 8;
  if (blocks > int64_t(h->num_sms) * 16) blocks = int64_t(h->num_sms) * 16;
  fde_finalize_kernel<<<int(blocks), 256, 0, s>>>(fde, n, h->fde_dim, static_cast<__nv_bfloat16*>(out_rows), inv_norm);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "launch fde_finalize");
}

static int launch_fde_scan_simt(b200ms_t* h, const void* F, const float* inv_norm, int64_t n_pages, const float* q_fde, int n_q,
                                float* scores, int64_t ld, cudaStream_t s) {
  const int nq_res = n_q < kFdeQ ? n_q : kFdeQ;  // queries resident per launch
  const size_t smem = size_t(nq_res) * h->fde_dim * sizeof(float);
  if (int e = ensure_smem(h, reinterpret_cast<const void*>(fde_scan_kernel), int(smem), "cudaFuncSetAttribute(fde_scan)"))
    return e;
  int per_sm = int((220 * 1024) / (smem + 1024));  // CTAs per SM by shared memory (40 KB per resident query)
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 8) per_sm = 8;
  int64_t blocks = (n_pages + 7) / 8;
  if (blocks > int64_t(h->num_sms) * per_sm) blocks = int64_t(h->num_sms) * per_sm;
  for (int qb = 0; qb < n_q; qb += kFdeQ) {
    fde_scan_kernel<<<int(blocks), 256, smem, s>>>(static_cast<const uint4*>(F), inv_norm, n_pages, h->fde_dim, q_fde, n_q, qb,
                                                   scores, ld);
    h->launches++;
    if (int e = check_cuda(h, cudaGetLastError(), "launch fde_scan")) return e;
  }
  return B200MS_OK;
}

int launch_fde_scan(b200ms_t* h, const void* F, const float* inv_norm, int64_t n_pages, const float* q_fde, int n_q,
                    float* scores, int64_t ld, cudaStream_t s) {
  if (n_pages <= 0 || n_q <= 0) return B200MS_OK;
  const int fd = h->fde_dim;
  const bool tensor = h->fde_gemm && fd % 64 == 0 && (reinterpret_cast<uintptr_t>(F) & 127) == 0 && n_pages >= 128;
  if (!tensor) {
    if (fd % 8) return set_error(h, B200MS_EINVAL, "fde_scan: fde_dim must be a multiple of 8");
    return launch_fde_scan_simt(h, F, inv_norm, n_pages, q_fde, n_q, scores, ld, s);
  }
  CUtensorMap tf;
  if (int e = make_tmap_rows(h, &tf, F, B200MS_BF16, n_pages, 128, int64_t(fd) * 2)) return e;
  for (int qb = 0; qb < n_q; qb += 128) {
    const int n_here = n_q - qb < 128 ? n_q - qb : 128;
    const int half = n_here <= 16 ? 16 : ((n_here + 31) & ~31);
    const int nqp = 2 * half;
    if (int e = reserve(h, h->fde_q_bf16, size_t(nqp) * fd * 2 + 1024)) return e;
    __nv_bfloat16* qb16 = reinterpret_cast<__nv_bfloat16*>((reinterpret_cast<uintptr_t>(h->fde_q_bf16.p) + 1023) & ~uintptr_t(1023));
    fde_q_split_kernel<<<h->num_sms, 256, 0, s>>>(q_fde + int64_t(qb) * fd, n_here, fd, half, qb16);
    h->launches++;
    if (int e = check_cuda(h, cudaGetLastError(), "launch fde_q_split")) return e;
    CUtensorMap tq;
    if (int e = make_tmap_rows(h, &tq, qb16, B200MS_BF16, nqp, nqp, int64_t(fd) * 2)) return e;
    const int n_tiles = int((n_pages + 127) / 128);
    if (int e = launch_persistent(h, fde_scan_umma_kernel, "fde_scan_umma", kScanThreads, 0, kScanATile + uint32_t(nqp) * 128u,
                                  12, n_tiles, s, tf, tq, inv_norm, n_pages, fd / 64, n_here, qb, half, scores, ld))
      return e;
  }
  return B200MS_OK;
}

}  // namespace bms

using namespace bms;

#define B200MS_API extern "C" __attribute__((visibility("default")))

// ------------------------------------------------------------------------------------------------ C-ABI
B200MS_API int b200ms_fde_configure(b200ms_t* h, int reps, int ksim, int proj_dim, float scale, const float* simhash,
                                    const int32_t* ams_index, const float* ams_sign) {
  return b200ms_fde_configure_ex(h, reps, ksim, proj_dim, scale, simhash, ams_index, ams_sign, 0, 0, nullptr, nullptr);
}

B200MS_API int b200ms_fde_configure_ex(b200ms_t* h, int reps, int ksim, int proj_dim, float scale, const float* simhash,
                                       const int32_t* ams_index, const float* ams_sign, int fill_empty_partitions,
                                       int final_dim, const int32_t* final_index, const float* final_sign) {
  if (!h) return B200MS_EINVAL;
  if (reps < 1 || ksim < 1 || ksim > 8 || proj_dim < 1 || proj_dim > 64 || (proj_dim << ksim) > 512 || ((proj_dim << ksim) % 8) ||
      !simhash || !ams_index || !ams_sign)
    return set_error(h, B200MS_EINVAL, "fde_configure: need 1<=ksim<=8, proj_dim<=64, proj_dim*2^ksim <= 512 and a multiple of 8");
  for (int i = 0; i < reps * kDim; ++i)
    if (ams_index[i] < 0 || ams_index[i] >= proj_dim) return set_error(h, B200MS_EINVAL, "fde_configure: ams_index out of range");
  const int inner = reps * (1 << ksim) * proj_dim;
  if (final_dim < 0 || (final_dim > 0 && (!final_index || !final_sign || final_dim % 8)))
    return set_error(h, B200MS_EINVAL, "fde_configure: final projection needs index/sign arrays and a dimension that is a multiple of 8");
  DeviceGuard g(h->device);
  cudaStream_t s = h->stream;
  if (int e = upload(h, h->fde_simhash, simhash, size_t(reps) * kDim * ksim * 4, s)) return e;
  if (int e = upload(h, h->fde_ams_index, ams_index, size_t(reps) * kDim * 4, s)) return e;
  if (int e = upload(h, h->fde_ams_sign, ams_sign, size_t(reps) * kDim * 4, s)) return e;
  if (final_dim > 0) {
    // CSR by output bucket, ascending input index inside a bucket (the order the oracle adds in)
    std::vector<int32_t> csr(size_t(final_dim) + 1 + size_t(inner), 0);
    std::vector<float> sg(static_cast<size_t>(inner), 0.f);
    for (int i = 0; i < inner; ++i) {
      if (final_index[i] < 0 || final_index[i] >= final_dim) return set_error(h, B200MS_EINVAL, "fde_configure: final_index out of range");
      csr[size_t(final_index[i]) + 1]++;
    }
    for (int j = 0; j < final_dim; ++j) csr[size_t(j) + 1] += csr[size_t(j)];
    std::vector<int32_t> fill(static_cast<size_t>(final_dim), 0);
    for (int i = 0; i < inner; ++i) {
      const int j = final_index[i];
      const size_t pos = size_t(csr[size_t(j)]) + size_t(fill[size_t(j)]++);
      csr[size_t(final_dim) + 1 + pos] = i;
      sg[pos] = final_sign[i];
    }
    if (int e = upload(h, h->fde_final_index, csr.data(), csr.size() * 4, s)) return e;
    if (int e = upload(h, h->fde_final_sign, sg.data(), sg.size() * 4, s)) return e;
  }
  if (int e = check_cuda(h, cudaStreamSynchronize(s), "fde_configure: sync")) return e;
  h->fde_reps = reps;
  h->fde_ksim = ksim;
  h->fde_proj = proj_dim;
  h->fde_scale = scale;
  h->fde_fill_empty = fill_empty_partitions ? 1 : 0;
  h->fde_inner_dim = inner;
  h->fde_dim = final_dim > 0 ? final_dim : inner;
  return B200MS_OK;
}

B200MS_API int64_t b200ms_fde_dim(const b200ms_t* h) { return h ? h->fde_dim : 0; }

// encode (+ optional final count-sketch projection) of n_items items described by item_start (+ item_len) on the device
static int encode_and_project(b200ms_t* h, const void* rows, int src_dtype, const int64_t* st_dev, const int32_t* len_dev,
                              int64_t n_items, int is_document, float* out, cudaStream_t s) {
  if (h->fde_dim == h->fde_inner_dim) return launch_fde_encode(h, rows, src_dtype, st_dev, int(n_items), is_document, out, s, len_dev);
  if (int e = reserve(h, h->fde_tmp, size_t(n_items) * size_t(h->fde_inner_dim) * 4)) return e;
  float* tmp = static_cast<float*>(h->fde_tmp.p);
  if (int e = launch_fde_encode(h, rows, src_dtype, st_dev, int(n_items), is_document, tmp, s, len_dev)) return e;
  int64_t blocks = (n_items * h->fde_dim + 255) / 256;
  if (blocks > int64_t(h->num_sms) * 16) blocks = int64_t(h->num_sms) * 16;
  fde_final_project_kernel<<<int(blocks), 256, 0, s>>>(tmp, n_items, h->fde_inner_dim, h->fde_dim,
                                                      static_cast<const int32_t*>(h->fde_final_index.p),
                                                      static_cast<const float*>(h->fde_final_sign.p), out);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "launch fde_final_project");
}

B200MS_API int b200ms_fde_encode(b200ms_t* h, const void* rows, int src_dtype, const int32_t* item_lens, int64_t n_items,
                                 int is_document, float* out, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (h->fde_dim == 0) return set_error(h, B200MS_ESTATE, "fde_encode: call b200ms_fde_configure first");
  if ((src_dtype != B200MS_F32 && src_dtype != B200MS_BF16) || n_items < 0 || n_items > 65535 ||
      (n_items > 0 && (!rows || !item_lens || !out)))
    return set_error(h, B200MS_EINVAL, "fde_encode: bad arguments (at most 65535 items per call)");
  if (n_items == 0) return B200MS_OK;
  DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  std::vector<int64_t> st(size_t(n_items) + 1);
  st[0] = 0;
  for (int64_t i = 0; i < n_items; ++i) st[i + 1] = st[i] + (item_lens[i] > 0 ? item_lens[i] : 0);
  if (int e = upload(h, h->meta_b, st.data(), st.size() * 8, s)) return e;
  return encode_and_project(h, rows, src_dtype, static_cast<const int64_t*>(h->meta_b.p), nullptr, n_items, is_document, out, s);
}

// Document FDEs of pages [first_page, first_page + n_pages) of the ATTACHED bf16 corpus, read from its packed rows (true
// page lengths; the padding rows are skipped) -- rebuilds the FDE matrix of a corpus loaded from a shard file without the
// float sources (SURVEY 8f-2).  The packed rows are the bf16 rounding of what was ingested; ColPali embeddings are bf16 to
// begin with (fast_multivector_store.py:674), so this reproduces the ingest-time encodings.
B200MS_API int b200ms_fde_encode_corpus(b200ms_t* h, int64_t first_page, int64_t n_pages, float* out, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (h->fde_dim == 0) return set_error(h, B200MS_ESTATE, "fde_encode_corpus: call b200ms_fde_configure first");
  const Corpus& c = h->corpus;
  if (c.dtype != B200MS_BF16) return set_error(h, B200MS_ESTATE, "fde_encode_corpus: needs an attached bf16 corpus");
  if (first_page < 0 || n_pages < 0 || n_pages > 65535 || first_page + n_pages > c.n_pages || (n_pages > 0 && !out))
    return set_error(h, B200MS_EINVAL, "fde_encode_corpus: bad page range (at most 65535 pages per call)");
  if (n_pages == 0) return B200MS_OK;
  DeviceGuard g(h->device);
  return encode_and_project(h, c.rows, B200MS_BF16, static_cast<const int64_t*>(h->page_start.p) + first_page,
                            static_cast<const int32_t*>(h->page_len.p) + first_page, n_pages, 1, out,
                            static_cast<cudaStream_t>(stream));
}

B200MS_API int b200ms_fde_finalize(b200ms_t* h, const float* fde, int64_t n, void* out_rows, float* inv_norm, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (h->fde_dim == 0) return set_error(h, B200MS_ESTATE, "fde_finalize: call b200ms_fde_configure first");
  if (n < 0 || (n > 0 && (!fde || !out_rows || !inv_norm))) return set_error(h, B200MS_EINVAL, "fde_finalize: bad arguments");
  DeviceGuard g(h->device);
  return launch_fde_finalize(h, fde, n, out_rows, inv_norm, static_cast<cudaStream_t>(stream));
}

B200MS_API int b200ms_fde_scan(b200ms_t* h, const void* fde_rows, const float* inv_norm, int64_t n_pages, const float* q_fde,
                               int n_q, float* scores, int64_t ld, void* stream) {
  if (!h) return B200MS_EINVAL;
  if (h->fde_dim == 0) return set_error(h, B200MS_ESTATE, "fde_scan: call b200ms_fde_configure first");
  if (n_pages < 0 || n_q < 0 || ld < n_pages || (n_pages > 0 && n_q > 0 && (!fde_rows || !inv_norm || !q_fde || !scores)) ||
      (reinterpret_cast<uintptr_t>(fde_rows) & 15))
    return set_error(h, B200MS_EINVAL, "fde_scan: bad arguments (rows 16-byte aligned, ld >= n_pages)");
  DeviceGuard g(h->device);
  return launch_fde_scan(h, fde_rows, inv_norm, n_pages, q_fde, n_q, scores, ld, static_cast<cudaStream_t>(stream));
}
