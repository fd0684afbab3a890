// Valid-row compaction for the Stage-2 head.  Rows whose mask weight is zero (and the never-scored last position of
// every sequence) contribute nothing to the loss or to any gradient (SURVEY.md Appendix A); with the reference's
// tokenisation (padding="max_length", 128 positions, 10-20 real tokens: pkg/data/preprocessing.py:223-231) that is
// > 80 % of the rows of a real Stage-2 batch.  These kernels build the list of scored rows, gather them (casting to the
// bf16 tensor-core operand on the way) into a dense [n][d] matrix, and scatter per-row results back.  All HBM-bound.
#include <initializer_list>

#include "common.h"
#include "ptx.cuh"

namespace pgica {
namespace {

// One block: index[0..count) = the rows r (ascending) with row_weight[r] != 0 (NaN weights count as scored: they must
// poison the sequence like in the reference), count[0] = how many.  Ballot + popc scan, 1024 rows per iteration.
__global__ void compact_rows_kernel(const float* __restrict__ row_weight, int rows, int* __restrict__ index,
                                    int* __restrict__ count) {
  __shared__ int warp_total[32];
  __shared__ int base_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) base_s = 0;
  __syncthreads();
  for (int start = 0; start < rows; start += 1024) {
    const int r = start + threadIdx.x;
    const bool valid = r < rows && row_weight[r] != 0.f;
    const unsigned ballot = __ballot_sync(0xffffffffu, valid);
    const int before = __popc(ballot & ((1u << lane) - 1u));
    if (lane == 0) warp_total[warp] = __popc(ballot);
    __syncthreads();
    int offset = base_s;
    for (int w = 0; w < warp; ++w) offset += warp_total[w];
    if (valid) index[offset + before] = r;
    __syncthreads();
    if (threadIdx.x == 1023) base_s = offset + before + (valid ? 1 : 0);
    __syncthreads();
  }
  if (threadIdx.x == 0) count[0] = base_s;
}

// o[0..d) = bf16(s[0..d)) (fp32 source: cast; bf16 source: 16-byte copies); the block's threads stride the row.
template <typename T>
__device__ __forceinline__ void cast_row_bf16(const T* __restrict__ s, __nv_bfloat16* __restrict__ o, int d) {
  if constexpr (sizeof(T) == 4) {
    for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
      const float4 v = *reinterpret_cast<const float4*>(s + c);
      __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
      uint2 p;
      p.x = *reinterpret_cast<unsigned*>(&lo);
      p.y = *reinterpret_cast<unsigned*>(&hi);
      *reinterpret_cast<uint2*>(o + c) = p;
    }
  } else {
    for (int c = threadIdx.x * 8; c < d; c += blockDim.x * 8)
      *reinterpret_cast<uint4*>(o + c) = *reinterpret_cast<const uint4*>(s + c);
  }
}

// dst[i][:] = bf16(src[index[i]][:]); optionally label_out[i] = label_in[index[i]].  One block per output row.
template <typename T>
__global__ void gather_rows_kernel(const T* __restrict__ src, const int* __restrict__ index, int d,
                                   __nv_bfloat16* __restrict__ dst, const int* __restrict__ label_in,
                                   int* __restrict__ label_out) {
  const int i = blockIdx.x;
  const int r = index[i];
  if (threadIdx.x == 0 && label_in) label_out[i] = label_in[r];
  cast_row_bf16(src + (size_t)r * d, dst + (size_t)i * d, d);
}

// o[0..d) = s[0..d) with a dtype change if asked (d % 4 == 0); s == nullptr writes zeros.
template <typename S, typename D>
__device__ __forceinline__ void convert_row(const S* __restrict__ s, D* __restrict__ o, int d) {
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (s == nullptr) {
    } else if constexpr (sizeof(S) == 4) {
      const float4 q = *reinterpret_cast<const float4*>(s + c);
      v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
    } else {
      const uint2 q = *reinterpret_cast<const uint2*>(s + c);
      const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&q.x);
      const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&q.y);
      v[0] = __low2float(a), v[1] = __high2float(a), v[2] = __low2float(b), v[3] = __high2float(b);
    }
    if constexpr (sizeof(D) == 4) {
      *reinterpret_cast<float4*>(o + c) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
      uint2 p;
      p.x = *reinterpret_cast<unsigned*>(&lo);
      p.y = *reinterpret_cast<unsigned*>(&hi);
      *reinterpret_cast<uint2*>(o + c) = p;
    }
  }
}

// dst[index[i]][:] = src[i][:] with a dtype change if asked (dst was zero-filled by the caller of the kernel)
template <typename S, typename D>
__global__ void scatter_rows_kernel(const S* __restrict__ src, const int* __restrict__ index, int d,
                                    D* __restrict__ dst) {
  const int i = blockIdx.x;
  convert_row(src + (size_t)i * d, dst + (size_t)index[i] * d, d);
}

// 4-byte elements (float or int32 bit patterns): dst[i] = src[index[i]]  /  dst[index[i]] = src[i]
__global__ void gather_u32_kernel(const unsigned* __restrict__ src, const int* __restrict__ index, int n,
                                  unsigned* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[index[i]];
}
__global__ void scatter_u32_kernel(const unsigned* __restrict__ src, const int* __restrict__ index, int n,
                                   unsigned* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[index[i]] = src[i];
}


// ---- device-count forms: the row count stays on the device, launches are sized by the caller's rows_launch >= n ----
// Every index is range-checked before use: a row count larger than rows_launch (masks that disagree with the caller's
// bucket) only drops rows and raises the overflow flag, it never reads or writes outside a buffer.

struct RowSets {
  int nset;
  int begin[PGICA_COMPACT_MAX_SETS + 1];  // set s owns rows [begin[s], begin[s + 1]) of the concatenated row space
  const void* src[PGICA_COMPACT_MAX_SETS];
  int src_is_bf16[PGICA_COMPACT_MAX_SETS];
};

// One block of 1024 threads.  slot[r] = position of row r among the scored rows of all sets (ascending), -1 when row r is
// not scored; index[p] = r for p < min(n, rows_launch), -1 for the padding positions [n, rows_launch).
// info = {counts[nset], offsets[nset], n, overflow}.
__global__ void __launch_bounds__(1024) compact_rows_dev_kernel(const float* __restrict__ row_weight, RowSets sets,
                                                                int rows_launch, int* __restrict__ index,
                                                                int* __restrict__ slot, int* __restrict__ info) {
  __shared__ int warp_total[32];
  __shared__ int base_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nset = sets.nset, rows = sets.begin[nset];
  if (threadIdx.x == 0) base_s = 0;
  __syncthreads();
  for (int start = 0; start < rows; start += 1024) {
    const int r = start + threadIdx.x;
    const bool valid = r < rows && row_weight[r] != 0.f;
    const unsigned ballot = __ballot_sync(0xffffffffu, valid);
    const int before = __popc(ballot & ((1u << lane) - 1u));
    if (lane == 0) warp_total[warp] = __popc(ballot);
    __syncthreads();
    int pos = base_s + before;
    for (int w = 0; w < warp; ++w) pos += warp_total[w];
    if (r < rows) {
      slot[r] = valid ? pos : -1;
      if (valid && pos < rows_launch) index[pos] = r;
      for (int s = 0; s < nset; ++s)
        if (r == sets.begin[s]) info[nset + s] = pos;  // scored rows before set s
    }
    __syncthreads();
    if (threadIdx.x == 1023) base_s = pos + (valid ? 1 : 0);
    __syncthreads();
  }
  const int n = base_s;
  for (int p = n + threadIdx.x; p < rows_launch; p += blockDim.x) index[p] = -1;
  if (threadIdx.x < nset) {
    const int s = threadIdx.x;
    info[s] = (s + 1 < nset ? info[nset + s + 1] : n) - info[nset + s];
  }
  if (threadIdx.x == 0) {
    info[2 * nset] = n;
    info[2 * nset + 1] = n > rows_launch ? 1 : 0;
  }
}

// dst[i][:] = bf16(row index[i] of its set's source), label_out[i] = label_in[index[i]] (when given); a padding position
// (index outside [0, rows)) gets a zero row and label -1.  One block per position of [0, rows_launch).
__global__ void gather_rows_dev_kernel(RowSets sets, const int* __restrict__ index, int d,
                                       __nv_bfloat16* __restrict__ dst, const int* __restrict__ label_in,
                                       int* __restrict__ label_out) {
  const int i = blockIdx.x;
  const int r = index[i];
  __nv_bfloat16* o = dst + (size_t)i * d;
  if (r < 0 || r >= sets.begin[sets.nset]) {
    if (threadIdx.x == 0 && label_out) label_out[i] = -1;
    for (int c = threadIdx.x * 8; c < d; c += blockDim.x * 8) *reinterpret_cast<uint4*>(o + c) = make_uint4(0, 0, 0, 0);
    return;
  }
  int s = 0;
  while (s + 1 < sets.nset && r >= sets.begin[s + 1]) ++s;
  if (threadIdx.x == 0 && label_out) label_out[i] = label_in[r];
  const size_t off = (size_t)(r - sets.begin[s]) * d;
  if (sets.src_is_bf16[s])
    cast_row_bf16(static_cast<const __nv_bfloat16*>(sets.src[s]) + off, o, d);
  else
    cast_row_bf16(static_cast<const float*>(sets.src[s]) + off, o, d);
}

// dst[i] = src[index[i]] for 0 <= index[i] < src_n, else 0 (padding positions get a zero coefficient)
__global__ void gather_u32_dev_kernel(const unsigned* __restrict__ src, int src_n, const int* __restrict__ index,
                                      int n, unsigned* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int r = index[i];
  dst[i] = (r >= 0 && r < src_n) ? src[r] : 0u;
}

// dst[r] = src[slot[r]] for 0 <= slot[r] < src_n; 0 for an unscored row (slot < 0); a quiet NaN for a scored row that did
// not fit the launch (slot >= src_n), so that the sequence it belongs to, and the loss, become NaN.
__global__ void scatter_u32_dev_kernel(const unsigned* __restrict__ src, int src_n, const int* __restrict__ slot,
                                       int rows, unsigned* __restrict__ dst) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int p = slot[r];
  dst[r] = p < 0 ? 0u : (p < src_n ? src[p] : 0x7fc00000u);
}

// dst[r][:] = src[slot[r]][:] for 0 <= slot[r] < src_n, else zeros.  One block per destination row: every row is written.
template <typename S, typename D>
__global__ void scatter_rows_dev_kernel(const S* __restrict__ src, int src_n, const int* __restrict__ slot, int d,
                                        D* __restrict__ dst) {
  const int r = blockIdx.x;
  const int p = slot[r];
  convert_row((p >= 0 && p < src_n) ? src + (size_t)p * d : nullptr, dst + (size_t)r * d, d);
}

}  // namespace
}  // namespace pgica

namespace pgica {
namespace {
// PGICA_OK when every non-null pointer is device (or managed) memory: a host pointer handed to a kernel would fault.
int require_device(const char* what, std::initializer_list<const void*> ptrs) {
  for (const void* p : ptrs) {
    if (!p) continue;
    cudaPointerAttributes a;
    const cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      set_error("%s: cannot query pointer %p: %s", what, p, cudaGetErrorString(e));
      return PGICA_ERR_INVALID_ARGUMENT;
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) {
      set_error("%s: %p is not device memory", what, p);
      return PGICA_ERR_INVALID_ARGUMENT;
    }
  }
  return PGICA_OK;
}

// Row sets from the host arrays of the device-count entry points; total rows in [1, 2^31).
int make_row_sets(const char* what, int nset, const int64_t* rows_host, RowSets* sets) {
  PGICA_REQUIRE(nset >= 1 && nset <= PGICA_COMPACT_MAX_SETS && rows_host, "%s: need 1..%d sets (got %d)", what,
                PGICA_COMPACT_MAX_SETS, nset);
  *sets = RowSets{};
  sets->nset = nset;
  int64_t total = 0;
  for (int s = 0; s < nset; ++s) {
    PGICA_REQUIRE(rows_host[s] > 0, "%s: set %d has %lld rows", what, s, (long long)rows_host[s]);
    sets->begin[s] = (int)total;
    total += rows_host[s];
    PGICA_REQUIRE(total < (1ll << 31), "%s: too many rows", what);
  }
  sets->begin[nset] = (int)total;
  return PGICA_OK;
}
}  // namespace
}  // namespace pgica

extern "C" {

using namespace pgica;

int pgica_compact_rows(const float* row_weight, int64_t rows, int32_t* index, int32_t* count, void* stream) {
  PGICA_REQUIRE(row_weight && index && count, "compact_rows: null pointer");
  PGICA_REQUIRE(rows > 0 && rows < (1ll << 31), "compact_rows: bad row count");
  compact_rows_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(row_weight, (int)rows, index, count);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_gather_rows_bf16(const void* src, int src_is_bf16, const int32_t* index, int64_t n, int64_t d,
                           void* dst_bf16, const int32_t* label_in, int32_t* label_out, void* stream) {
  PGICA_REQUIRE(src && index && dst_bf16, "gather_rows: null pointer");
  PGICA_REQUIRE((label_in == nullptr) == (label_out == nullptr), "gather_rows: labels come as an in/out pair");
  PGICA_REQUIRE(n >= 0 && n < (1ll << 31) && d > 0 && d % 8 == 0, "gather_rows: need d %% 8 == 0 (got n %lld, d %lld)",
                (long long)n, (long long)d);
  PGICA_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst_bf16)) & 15u) == 0,
                "gather_rows: pointers must be 16-byte aligned");
  if (n == 0) return PGICA_OK;
  const int threads = d >= 1024 ? 256 : 128;
  if (src_is_bf16)
    gather_rows_kernel<__nv_bfloat16><<<(unsigned)n, threads, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(src), index, (int)d, static_cast<__nv_bfloat16*>(dst_bf16), label_in,
        label_out);
  else
    gather_rows_kernel<float><<<(unsigned)n, threads, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(src), index, (int)d, static_cast<__nv_bfloat16*>(dst_bf16), label_in, label_out);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_scatter_rows(const void* src, int src_is_bf16, const int32_t* index, int64_t n, int64_t d, void* dst,
                       int dst_is_bf16, int64_t dst_rows, void* stream) {
  PGICA_REQUIRE(src && index && dst, "scatter_rows: null pointer");
  PGICA_REQUIRE(n >= 0 && n <= dst_rows && dst_rows < (1ll << 31) && d > 0 && d % 4 == 0,
                "scatter_rows: bad shape (n %lld, rows %lld, d %lld)", (long long)n, (long long)dst_rows, (long long)d);
  PGICA_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0,
                "scatter_rows: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  PGICA_CUDA_OK(cudaMemsetAsync(dst, 0, (size_t)dst_rows * d * (dst_is_bf16 ? 2 : 4), st));
  if (n == 0) return PGICA_OK;
  const unsigned g = (unsigned)n;
  const int dd = (int)d;
  if (src_is_bf16 && dst_is_bf16)
    scatter_rows_kernel<<<g, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(src), index, dd,
                                           static_cast<__nv_bfloat16*>(dst));
  else if (src_is_bf16)
    scatter_rows_kernel<<<g, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(src), index, dd, static_cast<float*>(dst));
  else if (dst_is_bf16)
    scatter_rows_kernel<<<g, 256, 0, st>>>(static_cast<const float*>(src), index, dd, static_cast<__nv_bfloat16*>(dst));
  else
    scatter_rows_kernel<<<g, 256, 0, st>>>(static_cast<const float*>(src), index, dd, static_cast<float*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_gather_u32(const void* src, const int32_t* index, int64_t n, void* dst, void* stream) {
  PGICA_REQUIRE(src && index && dst && n >= 0 && n < (1ll << 31), "gather_u32: bad argument");
  if (n == 0) return PGICA_OK;
  gather_u32_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const unsigned*>(src), index, (int)n, static_cast<unsigned*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_scatter_u32(const void* src, const int32_t* index, int64_t n, void* dst, int64_t dst_n, void* stream) {
  PGICA_REQUIRE(src && index && dst && n >= 0 && n <= dst_n && dst_n < (1ll << 31), "scatter_u32: bad argument");
  PGICA_CUDA_OK(cudaMemsetAsync(dst, 0, (size_t)dst_n * 4, (cudaStream_t)stream));
  if (n == 0) return PGICA_OK;
  scatter_u32_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const unsigned*>(src), index, (int)n, static_cast<unsigned*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_compact_rows_dev(const float* row_weight, int nset, const int64_t* rows_host, int64_t rows_launch,
                           int32_t* index, int32_t* slot, int32_t* info, void* stream) {
  RowSets sets;
  int rc = make_row_sets("compact_rows_dev", nset, rows_host, &sets);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(rows_launch > 0 && rows_launch < (1ll << 31), "compact_rows_dev: bad rows_launch %lld",
                (long long)rows_launch);
  PGICA_REQUIRE(row_weight && index && slot && info, "compact_rows_dev: null pointer");
  rc = require_device("compact_rows_dev", {row_weight, index, slot, info});
  if (rc != PGICA_OK) return rc;
  compact_rows_dev_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(row_weight, sets, (int)rows_launch, index, slot, info);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_gather_rows_bf16_dev(int nset, const void* const* src_host, const int32_t* src_is_bf16_host,
                               const int64_t* rows_host, const int32_t* index, int64_t rows_launch, int64_t d,
                               void* dst_bf16, const int32_t* label_in, int32_t* label_out, void* stream) {
  RowSets sets;
  int rc = make_row_sets("gather_rows_dev", nset, rows_host, &sets);
  if (rc != PGICA_OK) return rc;
  PGICA_REQUIRE(src_host && src_is_bf16_host && index && dst_bf16, "gather_rows_dev: null pointer");
  PGICA_REQUIRE((label_in == nullptr) == (label_out == nullptr), "gather_rows_dev: labels come as an in/out pair");
  PGICA_REQUIRE(rows_launch > 0 && rows_launch < (1ll << 31) && d > 0 && d % 8 == 0,
                "gather_rows_dev: need rows_launch > 0 and d %% 8 == 0 (got %lld, %lld)", (long long)rows_launch,
                (long long)d);
  uintptr_t align = reinterpret_cast<uintptr_t>(dst_bf16);
  for (int s = 0; s < nset; ++s) {
    PGICA_REQUIRE(src_host[s], "gather_rows_dev: null source of set %d", s);
    sets.src[s] = src_host[s];
    sets.src_is_bf16[s] = src_is_bf16_host[s] ? 1 : 0;
    align |= reinterpret_cast<uintptr_t>(src_host[s]);
    rc = require_device("gather_rows_dev", {src_host[s]});
    if (rc != PGICA_OK) return rc;
  }
  PGICA_REQUIRE((align & 15u) == 0, "gather_rows_dev: pointers must be 16-byte aligned");
  rc = require_device("gather_rows_dev", {index, dst_bf16, label_in, label_out});
  if (rc != PGICA_OK) return rc;
  gather_rows_dev_kernel<<<(unsigned)rows_launch, d >= 1024 ? 256 : 128, 0, (cudaStream_t)stream>>>(
      sets, index, (int)d, static_cast<__nv_bfloat16*>(dst_bf16), label_in, label_out);
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_gather_u32_dev(const void* src, int64_t src_n, const int32_t* index, int64_t n, void* dst, void* stream) {
  PGICA_REQUIRE(src && index && dst, "gather_u32_dev: null pointer");
  PGICA_REQUIRE(src_n > 0 && src_n < (1ll << 31) && n > 0 && n < (1ll << 31), "gather_u32_dev: bad size (%lld, %lld)",
                (long long)src_n, (long long)n);
  int rc = require_device("gather_u32_dev", {src, index, dst});
  if (rc != PGICA_OK) return rc;
  gather_u32_dev_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const unsigned*>(src), (int)src_n, index, (int)n, static_cast<unsigned*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_scatter_u32_dev(const void* src, int64_t src_n, const int32_t* slot, int64_t rows, void* dst, void* stream) {
  PGICA_REQUIRE(src && slot && dst, "scatter_u32_dev: null pointer");
  PGICA_REQUIRE(src_n > 0 && src_n < (1ll << 31) && rows > 0 && rows < (1ll << 31),
                "scatter_u32_dev: bad size (%lld, %lld)", (long long)src_n, (long long)rows);
  int rc = require_device("scatter_u32_dev", {src, slot, dst});
  if (rc != PGICA_OK) return rc;
  scatter_u32_dev_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const unsigned*>(src), (int)src_n, slot, (int)rows, static_cast<unsigned*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

int pgica_scatter_rows_dev(const void* src, int src_is_bf16, int64_t src_n, const int32_t* slot, int64_t rows,
                           int64_t d, void* dst, int dst_is_bf16, void* stream) {
  PGICA_REQUIRE(src && slot && dst, "scatter_rows_dev: null pointer");
  PGICA_REQUIRE(src_n > 0 && src_n < (1ll << 31) && rows > 0 && rows < (1ll << 31) && d > 0 && d % 4 == 0,
                "scatter_rows_dev: bad shape (src %lld, rows %lld, d %lld)", (long long)src_n, (long long)rows,
                (long long)d);
  PGICA_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0,
                "scatter_rows_dev: pointers must be 16-byte aligned");
  int rc = require_device("scatter_rows_dev", {src, slot, dst});
  if (rc != PGICA_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = (unsigned)rows;
  const int sn = (int)src_n, dd = (int)d;
  if (src_is_bf16 && dst_is_bf16)
    scatter_rows_dev_kernel<<<g, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(src), sn, slot, dd,
                                               static_cast<__nv_bfloat16*>(dst));
  else if (src_is_bf16)
    scatter_rows_dev_kernel<<<g, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(src), sn, slot, dd,
                                               static_cast<float*>(dst));
  else if (dst_is_bf16)
    scatter_rows_dev_kernel<<<g, 256, 0, st>>>(static_cast<const float*>(src), sn, slot, dd,
                                               static_cast<__nv_bfloat16*>(dst));
  else
    scatter_rows_dev_kernel<<<g, 256, 0, st>>>(static_cast<const float*>(src), sn, slot, dd, static_cast<float*>(dst));
  PGICA_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return PGICA_OK;
}

}  // extern "C"
