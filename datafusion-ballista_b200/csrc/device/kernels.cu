// Auxiliary CUDA kernels (sm_100a): aggregate-table init/extraction, prefix sums, hash-partition
// rank + scatter (ShuffleWriter), gathers, string view <-> Arrow Utf8 conversion, hash-join
// build/probe, LSD radix sort, and the synthetic TPC-H generator.
//
// Reference operators these stand behind: BatchPartitioner / compute_partition_indices +
// interleave_record_batch (ballista/core/src/execution_plans/sort_shuffle/writer.rs:729-749,
// partitioned_batch_iterator.rs:102-123), HashJoinExec and SortExec [EXT, DataFusion 53.1]
// (wire surface ballista/core/proto/datafusion.proto:1134-1144, :1286-1292).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../common/hash.hpp"
#include "../common/tpch_gen.hpp"
#include "kernels.h"

namespace b200 {

typedef __int128 i128;
typedef unsigned __int128 u128;

static inline int grid_for(int64_t n, int block, int per_thread = 1) {
  int64_t g = (n + (int64_t)block * per_thread - 1) / ((int64_t)block * per_thread);
  if (g < 1) g = 1;
  if (g > 148 * 16) g = 148 * 16;  // grid-stride loops; a multiple of the SM count
  return (int)g;
}

// ------------------------------------------------------------------------------------------------
// Aggregate table
// ------------------------------------------------------------------------------------------------
__global__ void agg_table_init_kernel(AggTable T, AccKinds kinds) {
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < T.cap; i += (unsigned long long)gridDim.x * blockDim.x) {
    T.hash[i] = 0;
    T.state[i] = 0;
    T.lock[i] = 0;
    for (int a = 0; a < kinds.n; a++) {
      unsigned long long lo = 0, hi = 0;
      switch (kinds.kind[a]) {
        case ACC_MIN_I128: lo = ~0ull; hi = 0x7FFFFFFFFFFFFFFFull; break;
        case ACC_MAX_I128: lo = 0; hi = 0x8000000000000000ull; break;
        case ACC_MIN_F64: lo = 0x7FFFFFFFFFFFFFFFull; break;
        case ACC_MAX_F64: lo = 0x8000000000000000ull; break;
        default: break;
      }
      T.acc[((unsigned long long)a * T.cap + i) * 2 + 0] = lo;
      T.acc[((unsigned long long)a * T.cap + i) * 2 + 1] = hi;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *T.n_groups = 0;
}
void launch_agg_table_init(const AggTable& T, const AccKinds& kinds, cudaStream_t st) {
  agg_table_init_kernel<<<grid_for((int64_t)T.cap, 256), 256, 0, st>>>(T, kinds);
}

__device__ __forceinline__ i128 mk128(unsigned long long lo, unsigned long long hi) { return (i128)(((u128)hi << 64) | lo); }
__device__ __forceinline__ double f64_from_key(long long k) {
  long long x = k ^ (long long)((unsigned long long)(k >> 63) >> 1);
  return __longlong_as_double(x);
}

__device__ void store_typed_i64(void* data, uint8_t phys, unsigned long long pos, long long v) {
  switch (phys) {
    case PH_I8:
    case PH_U8:
    case PH_BOOL8: ((int8_t*)data)[pos] = (int8_t)v; break;
    case PH_I16:
    case PH_U16: ((int16_t*)data)[pos] = (int16_t)v; break;
    case PH_I32:
    case PH_U32: ((int32_t*)data)[pos] = (int32_t)v; break;
    default: ((long long*)data)[pos] = v;
  }
}

__global__ void agg_extract_kernel(AggTable T, AggExtractArgs A) {
  for (unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; s < T.cap; s += (unsigned long long)gridDim.x * blockDim.x) {
    if (T.state[s] != 2) continue;
    unsigned long long pos = atomicAdd(A.counter, 1ull);
    if (pos >= A.cap) continue;
    for (int j = 0; j < A.n_out; j++) {
      const AggOut& o = A.out[j];
      switch (o.kind) {
        case AO_KEY: {
          unsigned long long w0 = T.keys[((unsigned long long)o.a * T.cap + s) * 2 + 0];
          unsigned long long w1 = T.keys[((unsigned long long)o.a * T.cap + s) * 2 + 1];
          unsigned char v = T.key_valid[(unsigned long long)o.a * T.cap + s];
          if (o.phys == PH_DEC128 || o.phys == PH_STRVIEW) ((ulonglong2*)o.data)[pos] = make_ulonglong2(w0, w1);
          else if (o.phys == PH_F64) ((unsigned long long*)o.data)[pos] = w0;
          else if (o.phys == PH_F32) ((float*)o.data)[pos] = (float)__longlong_as_double((long long)w0);
          else store_typed_i64(o.data, o.phys, pos, (long long)w0);
          if (o.valid) o.valid[pos] = v;
          break;
        }
        case AO_KEY_PACKED: {
          unsigned long long w0 = T.keys[((unsigned long long)o.a * T.cap + s) * 2 + 0];
          unsigned char v = T.key_valid[(unsigned long long)o.a * T.cap + s];
          unsigned long long len = w0 >> o.imm;
          unsigned long long bytes = w0 & ((1ull << o.imm) - 1);
          unsigned long long* dst = (unsigned long long*)o.aux + pos;
          *dst = bytes;
          ((ulonglong2*)o.data)[pos] = make_ulonglong2(v ? (unsigned long long)dst : 0ull, v ? len : 0ull);
          if (o.valid) o.valid[pos] = v;
          break;
        }
        default: {
          unsigned long long lo = T.acc[((unsigned long long)o.a * T.cap + s) * 2 + 0];
          unsigned long long hi = T.acc[((unsigned long long)o.a * T.cap + s) * 2 + 1];
          unsigned long long cnt = o.b == 255 ? 1ull : T.acc[((unsigned long long)o.b * T.cap + s) * 2 + 0];
          bool ok = cnt > 0;
          switch (o.kind) {
            case AO_ACC_I128: ((ulonglong2*)o.data)[pos] = make_ulonglong2(lo, hi); break;
            case AO_ACC_I64: store_typed_i64(o.data, o.phys, pos, (long long)lo); break;
            case AO_ACC_F64: ((unsigned long long*)o.data)[pos] = lo; break;
            case AO_COUNT:
              store_typed_i64(o.data, o.phys, pos, (long long)lo);
              ok = true;
              break;
            case AO_MINMAX_F64: ((double*)o.data)[pos] = f64_from_key((long long)lo); break;
            case AO_AVG_DEC: {
              i128 sum = mk128(lo, hi);
              i128 res = 0;
              if (ok) {
                // DecimalAverager::avg [EXT]: sum * 10^imm / count, truncating; overflow is an error
                i128 mul = 1;
                for (int k = 0; k < o.imm; k++) mul *= 10;
                i128 lim = ((i128)1 << 126) / (mul > 0 ? mul : 1);
                if (sum > lim || sum < -lim) atomicMax(A.error, 1u);
                res = (sum * mul) / (i128)cnt;
              }
              ((ulonglong2*)o.data)[pos] = make_ulonglong2((unsigned long long)res, (unsigned long long)((u128)res >> 64));
              break;
            }
            case AO_AVG_F64: {
              double sum = __longlong_as_double((long long)lo);
              ((double*)o.data)[pos] = ok ? sum / (double)cnt : 0.0;
              break;
            }
            default: break;
          }
          if (o.valid) o.valid[pos] = ok ? 1 : 0;
        }
      }
    }
  }
}
void launch_agg_extract(const AggTable& T, const AggExtractArgs& A, cudaStream_t st) {
  agg_extract_kernel<<<grid_for((int64_t)T.cap, 256), 256, 0, st>>>(T, A);
}

// ------------------------------------------------------------------------------------------------
// Exclusive scan (3 kernels: block scan, scan of block totals, add)
// ------------------------------------------------------------------------------------------------
static const int SCAN_BLOCK = 256, SCAN_ITEMS = 4, SCAN_TILE = SCAN_BLOCK * SCAN_ITEMS;

__device__ __forceinline__ uint64_t block_exclusive_scan(uint64_t v, uint64_t* total, uint64_t* warp_sums /*[32]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint64_t y = __shfl_up_sync(0xFFFFFFFFu, w, o);
      if (lane >= o) w += y;
    }
    warp_sums[lane] = w;
  }
  __syncthreads();
  uint64_t base = warp ? warp_sums[warp - 1] : 0;
  *total = warp_sums[(blockDim.x >> 5) - 1];
  return base + x - v;
}

__global__ void scan_block_kernel(const uint32_t* in, uint64_t* out, int64_t n, uint64_t* block_sums) {
  __shared__ uint64_t ws[32];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  uint64_t v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    v[i] = (base + i < n) ? in[base + i] : 0;
    s += v[i];
  }
  uint64_t total;
  uint64_t ex = block_exclusive_scan(s, &total, ws);
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    if (base + i < n) out[base + i] = ex;
    ex += v[i];
  }
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}
__global__ void scan_sums_kernel(uint64_t* block_sums, int64_t nb, uint64_t* grand_total) {
  __shared__ uint64_t ws[32];
  __shared__ uint64_t carry_sh;
  if (threadIdx.x == 0) carry_sh = 0;
  __syncthreads();
  for (int64_t c = 0; c < nb; c += blockDim.x) {
    int64_t i = c + threadIdx.x;
    uint64_t v = i < nb ? block_sums[i] : 0;
    uint64_t total;
    uint64_t ex = block_exclusive_scan(v, &total, ws);
    uint64_t carry = carry_sh;
    if (i < nb) block_sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry_sh = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *grand_total = carry_sh;
}
__global__ void scan_add_kernel(uint64_t* out, int64_t n, const uint64_t* block_sums, const uint64_t* grand_total) {
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  uint64_t add = block_sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++)
    if (base + i < n) out[base + i] += add;
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *grand_total;
}
void launch_scan_u32_to_u64(const uint32_t* in, uint64_t* out, int64_t n, uint64_t* scratch, cudaStream_t st) {
  int64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (nb < 1) nb = 1;
  scan_block_kernel<<<(unsigned)nb, SCAN_BLOCK, 0, st>>>(in, out, n, scratch);
  scan_sums_kernel<<<1, 256, 0, st>>>(scratch, nb, scratch + nb);
  scan_add_kernel<<<(unsigned)nb, SCAN_BLOCK, 0, st>>>(out, n, scratch, scratch + nb);
}

// ------------------------------------------------------------------------------------------------
// Hash partition: histogram, rank, scatter
// ------------------------------------------------------------------------------------------------
__global__ void histogram_kernel(const uint32_t* ids, int64_t n, uint32_t n_bins, unsigned long long* counts) {
  extern __shared__ unsigned int sh[];
  const bool use_sh = n_bins <= 8192;
  if (use_sh) {
    for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x) sh[b] = 0;
    __syncthreads();
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (use_sh) atomicAdd(&sh[ids[i]], 1u);
    else atomicAdd(&counts[ids[i]], 1ull);
  }
  if (use_sh) {
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x)
      if (sh[b]) atomicAdd(&counts[b], (unsigned long long)sh[b]);
  }
}
void launch_histogram_u32(const uint32_t* ids, int64_t n, uint32_t n_bins, unsigned long long* counts, cudaStream_t st) {
  size_t sm = n_bins <= 8192 ? n_bins * sizeof(unsigned int) : 0;
  histogram_kernel<<<grid_for(n, 256, 8), 256, sm, st>>>(ids, n, n_bins, counts);
}

template <typename T>
__global__ void scatter_kernel(const T* in, T* out, const uint32_t* dest, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[dest[i]] = in[i];
}
void launch_scatter_fixed(const void* in, void* out, const uint32_t* dest, int64_t n, int width, cudaStream_t st) {
  int g = grid_for(n, 256, 4);
  switch (width) {
    case 1: scatter_kernel<uint8_t><<<g, 256, 0, st>>>((const uint8_t*)in, (uint8_t*)out, dest, n); break;
    case 2: scatter_kernel<uint16_t><<<g, 256, 0, st>>>((const uint16_t*)in, (uint16_t*)out, dest, n); break;
    case 4: scatter_kernel<uint32_t><<<g, 256, 0, st>>>((const uint32_t*)in, (uint32_t*)out, dest, n); break;
    case 8: scatter_kernel<uint64_t><<<g, 256, 0, st>>>((const uint64_t*)in, (uint64_t*)out, dest, n); break;
    default: scatter_kernel<ulonglong2><<<g, 256, 0, st>>>((const ulonglong2*)in, (ulonglong2*)out, dest, n); break;
  }
}

template <typename T>
__global__ void gather_kernel(const T* in, const uint8_t* valid_in, T* out, uint8_t* valid_out, const int64_t* idx, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t j = idx[i];
    T z;
    memset(&z, 0, sizeof(T));
    out[i] = j >= 0 ? in[j] : z;
    if (valid_out) valid_out[i] = j >= 0 ? (valid_in ? valid_in[j] : 1) : 0;
  }
}
void launch_gather_fixed(const void* in, const uint8_t* valid_in, void* out, uint8_t* valid_out, const int64_t* idx, int64_t n, int width, cudaStream_t st) {
  int g = grid_for(n, 256, 4);
  switch (width) {
    case 1: gather_kernel<uint8_t><<<g, 256, 0, st>>>((const uint8_t*)in, valid_in, (uint8_t*)out, valid_out, idx, n); break;
    case 2: gather_kernel<uint16_t><<<g, 256, 0, st>>>((const uint16_t*)in, valid_in, (uint16_t*)out, valid_out, idx, n); break;
    case 4: gather_kernel<uint32_t><<<g, 256, 0, st>>>((const uint32_t*)in, valid_in, (uint32_t*)out, valid_out, idx, n); break;
    case 8: gather_kernel<uint64_t><<<g, 256, 0, st>>>((const uint64_t*)in, valid_in, (uint64_t*)out, valid_out, idx, n); break;
    default: gather_kernel<ulonglong2><<<g, 256, 0, st>>>((const ulonglong2*)in, valid_in, (ulonglong2*)out, valid_out, idx, n); break;
  }
}
// ingest: sign-extend host-narrowed Decimal128 values (int32 / int64) back to 16 bytes
template <typename T>
__global__ void widen_to_i128_kernel(const T* in, ulonglong2* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const long long v = (long long)in[i];
    out[i] = make_ulonglong2((unsigned long long)v, (unsigned long long)(v >> 63));
  }
}
void launch_widen_to_i128(const void* in, int width, void* out, int64_t n, cudaStream_t st) {
  if (n <= 0) return;
  if (width == 4) widen_to_i128_kernel<int32_t><<<grid_for(n, 256, 4), 256, 0, st>>>((const int32_t*)in, (ulonglong2*)out, n);
  else widen_to_i128_kernel<int64_t><<<grid_for(n, 256, 4), 256, 0, st>>>((const int64_t*)in, (ulonglong2*)out, n);
}

// Arrow offsets of a row slice -> offsets starting at 0; also reports the slice's first/last offset
// (the chars range) without a host round trip per column
__global__ void rebase_offsets_kernel(const int32_t* in, int64_t n_plus_1, int32_t* out, int32_t* first_last) {
  const int32_t base = in[0];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_plus_1; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i] - base;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    first_last[0] = base;
    first_last[1] = in[n_plus_1 - 1];
  }
}
void launch_rebase_offsets(const int32_t* in, int64_t n_plus_1, int32_t* out, int32_t* first_last, cudaStream_t st) {
  rebase_offsets_kernel<<<grid_for(n_plus_1, 256, 4), 256, 0, st>>>(in, n_plus_1, out, first_last);
}

// every column of a batch in one launch (blockIdx.y = column): the tail of a query handles a few rows
// in a dozen columns and is bound by launch count, not bytes
template <typename T>
__device__ __forceinline__ void gather_one(const GatherCol& c, const int64_t* idx, int64_t i) {
  const int64_t j = idx[i];
  T z;
  memset(&z, 0, sizeof(T));
  ((T*)c.out)[i] = j >= 0 ? ((const T*)c.in)[j] : z;
}
__global__ void gather_multi_kernel(const GatherCols cols, const int64_t* idx, int64_t n) {
  const GatherCol& c = cols.c[blockIdx.y];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    switch (c.width) {
      case 1: gather_one<uint8_t>(c, idx, i); break;
      case 2: gather_one<uint16_t>(c, idx, i); break;
      case 4: gather_one<uint32_t>(c, idx, i); break;
      case 8: gather_one<uint64_t>(c, idx, i); break;
      default: gather_one<ulonglong2>(c, idx, i); break;
    }
    if (c.valid_out) {
      const int64_t j = idx[i];
      c.valid_out[i] = j >= 0 ? (c.valid_in ? c.valid_in[j] : 1) : 0;
    }
  }
}
void launch_gather_multi(const GatherCols& cols, const int64_t* idx, int64_t n, cudaStream_t st) {
  if (cols.n <= 0) return;
  dim3 grid((unsigned)grid_for(n, 256, 4), (unsigned)cols.n);
  gather_multi_kernel<<<grid, 256, 0, st>>>(cols, idx, n);
}
__global__ void iota_i64_kernel(int64_t* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = i;
}
void launch_iota_i64(int64_t* out, int64_t n, cudaStream_t st) { iota_i64_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(out, n); }
__global__ void iota_u32_kernel(uint32_t* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (uint32_t)i;
}
void launch_iota_u32(uint32_t* out, int64_t n, cudaStream_t st) { iota_u32_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(out, n); }
__global__ void u32_to_i64_kernel(const uint32_t* in, int64_t* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i];
}
void launch_u32_to_i64(const uint32_t* in, int64_t* out, int64_t n, cudaStream_t st) { u32_to_i64_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(in, out, n); }

// ------------------------------------------------------------------------------------------------
// Strings and validity
// ------------------------------------------------------------------------------------------------
__global__ void utf8_to_views_kernel(const int32_t* offsets, const uint8_t* chars, unsigned long long* views, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int32_t o0 = offsets[i], o1 = offsets[i + 1];
    views[2 * i] = (unsigned long long)(chars + o0);
    views[2 * i + 1] = (unsigned long long)(uint32_t)(o1 - o0);
  }
}
void launch_utf8_to_views(const int32_t* offsets, const uint8_t* chars, unsigned long long* views, int64_t n, cudaStream_t st) {
  utf8_to_views_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(offsets, chars, views, n);
}
// 32-bit images (len << 24 | up to 3 bytes, first character in the low byte: the OP_STR_PACK8 image) of a Utf8 column whose
// strings are all at most 3 bytes long -- the companion the fused aggregate kernel reads instead of offsets + characters
__global__ void prepack3_kernel(const int32_t* offsets, const uint8_t* chars, int64_t n, uint32_t* out, unsigned int* too_long) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t o0 = offsets[i];
    const uint32_t len = (uint32_t)(offsets[i + 1] - o0);
    uint32_t v = 0;
    if (len > 3) {
      *too_long = 1u;
    } else {
      for (uint32_t k = 0; k < len; k++) v |= (uint32_t)chars[o0 + k] << (8 * k);
      v |= len << 24;
    }
    out[i] = v;
  }
}
void launch_prepack3(const int32_t* offsets, const uint8_t* chars, int64_t n, uint32_t* out, unsigned int* too_long, cudaStream_t st) {
  prepack3_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(offsets, chars, n, out, too_long);
}
__global__ void view_lengths_kernel(const unsigned long long* views, const uint8_t* valid, uint32_t* lens, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    lens[i] = (valid && !valid[i]) ? 0u : (uint32_t)views[2 * i + 1];
}
void launch_view_lengths(const unsigned long long* views, const uint8_t* valid, uint32_t* lens, int64_t n, cudaStream_t st) {
  view_lengths_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(views, valid, lens, n);
}
__global__ void views_to_utf8_kernel(const unsigned long long* views, const uint8_t* valid, const uint64_t* offs64, int32_t* offsets_out,
                                     uint8_t* chars_out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
    offsets_out[i] = (int32_t)offs64[i];
    if (i == n) break;
    if (valid && !valid[i]) continue;
    const uint8_t* p = (const uint8_t*)views[2 * i];
    uint32_t len = (uint32_t)views[2 * i + 1];
    uint8_t* d = chars_out + offs64[i];
    for (uint32_t k = 0; k < len; k++) d[k] = p[k];
  }
}
void launch_views_to_utf8(const unsigned long long* views, const uint8_t* valid, const uint64_t* offs64, int32_t* offsets_out, uint8_t* chars_out,
                          int64_t n, cudaStream_t st) {
  views_to_utf8_kernel<<<grid_for(n + 1, 256, 2), 256, 0, st>>>(views, valid, offs64, offsets_out, chars_out, n);
}
__global__ void bitmap_to_bytes_kernel(const uint8_t* bitmap, int64_t bit_offset, uint8_t* bytes, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t b = i + bit_offset;
    bytes[i] = (bitmap[b >> 3] >> (b & 7)) & 1;
  }
}
void launch_bitmap_to_bytes(const uint8_t* bitmap, int64_t bit_offset, uint8_t* bytes, int64_t n, cudaStream_t st) {
  bitmap_to_bytes_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(bitmap, bit_offset, bytes, n);
}
__global__ void bytes_to_bitmap_kernel(const uint8_t* bytes, uint8_t* bitmap, int64_t n, unsigned long long* null_count) {
  // one thread per output byte
  int64_t nbytes = (n + 7) / 8;
  unsigned long long nulls = 0;
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < nbytes; b += (int64_t)gridDim.x * blockDim.x) {
    uint8_t v = 0;
    for (int k = 0; k < 8; k++) {
      int64_t i = b * 8 + k;
      if (i < n) {
        if (bytes[i]) v |= (uint8_t)(1u << k);
        else nulls++;
      }
    }
    bitmap[b] = v;
  }
  if (null_count && nulls) atomicAdd(null_count, nulls);
}
void launch_bytes_to_bitmap(const uint8_t* bytes, uint8_t* bitmap, int64_t n, unsigned long long* null_count, cudaStream_t st) {
  bytes_to_bitmap_kernel<<<grid_for((n + 7) / 8, 256, 1), 256, 0, st>>>(bytes, bitmap, n, null_count);
}

// ------------------------------------------------------------------------------------------------
// Hash join (bucket-chained table on the build side; two-pass probe: count -> scan -> write)
// ------------------------------------------------------------------------------------------------
__global__ void join_build_kernel(const uint64_t* build_hash, const uint8_t* build_ok, int64_t n, int32_t* heads, uint64_t mask, int32_t* next) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (build_ok && !build_ok[i]) {
      next[i] = -1;
      continue;
    }
    uint64_t b = mix64(build_hash[i]) & mask;
    next[i] = atomicExch(&heads[b], (int32_t)i);
  }
}
void launch_join_build(const uint64_t* build_hash, const uint8_t* build_ok, int64_t n_build, int32_t* heads, uint64_t n_buckets, int32_t* next,
                       cudaStream_t st) {
  join_build_kernel<<<grid_for(n_build, 256, 4), 256, 0, st>>>(build_hash, build_ok, n_build, heads, n_buckets - 1, next);
}

__device__ __forceinline__ bool key_cols_equal(const JoinKeys& K, int64_t bi, int64_t pi) {
  for (int k = 0; k < K.n_keys; k++) {
    const KeyCol& b = K.build[k];
    const KeyCol& p = K.probe[k];
    bool bv = !b.valid || b.valid[bi], pv = !p.valid || p.valid[pi];
    if (!bv || !pv) {
      if (K.null_equals_null && !bv && !pv) continue;
      return false;
    }
    if (b.phys == PH_STRVIEW) {
      const unsigned long long* x = (const unsigned long long*)b.data + 2 * bi;
      const unsigned long long* y = (const unsigned long long*)p.data + 2 * pi;
      if (x[1] != y[1]) return false;
      const uint8_t *s = (const uint8_t*)x[0], *t = (const uint8_t*)y[0];
      for (uint32_t i = 0; i < (uint32_t)x[1]; i++)
        if (s[i] != t[i]) return false;
    } else if (b.phys == PH_F64) {
      double x = ((const double*)b.data)[bi], y = ((const double*)p.data)[pi];
      if (!(x == y || (x != x && y != y))) return false;
    } else {
      const uint8_t* x = (const uint8_t*)b.data + bi * b.width;
      const uint8_t* y = (const uint8_t*)p.data + pi * p.width;
      switch (b.width) {
        case 16:
          if (((const uint64_t*)x)[0] != ((const uint64_t*)y)[0] || ((const uint64_t*)x)[1] != ((const uint64_t*)y)[1]) return false;
          break;
        case 8:
          if (*(const uint64_t*)x != *(const uint64_t*)y) return false;
          break;
        case 4:
          if (*(const uint32_t*)x != *(const uint32_t*)y) return false;
          break;
        case 2:
          if (*(const uint16_t*)x != *(const uint16_t*)y) return false;
          break;
        default:
          if (*x != *y) return false;
      }
    }
  }
  return true;
}

template <bool WRITE>
__global__ void join_probe_kernel(JoinKeys K, const uint64_t* build_hash, const int32_t* heads, uint64_t mask, const int32_t* next,
                                  const uint64_t* probe_hash, const uint8_t* probe_ok, int64_t n_probe, uint32_t* counts, uint8_t* build_mark,
                                  const uint64_t* offsets, int64_t* out_b, int64_t* out_p) {
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n_probe; j += (int64_t)gridDim.x * blockDim.x) {
    uint32_t c = 0;
    if (!probe_ok || probe_ok[j]) {
      const uint64_t h = probe_hash[j];
      uint64_t w = WRITE ? offsets[j] : 0;
      for (int32_t i = heads[mix64(h) & mask]; i >= 0; i = next[i]) {
        if (build_hash[i] != h) continue;
        if (!key_cols_equal(K, i, j)) continue;
        if (WRITE) {
          out_b[w] = i;
          out_p[w] = j;
          w++;
        } else {
          c++;
          if (build_mark) build_mark[i] = 1;
        }
      }
    }
    if (!WRITE) counts[j] = c;
  }
}
void launch_join_probe_count(const JoinKeys& K, const uint64_t* build_hash, const int32_t* heads, uint64_t n_buckets, const int32_t* next,
                             const uint64_t* probe_hash, const uint8_t* probe_ok, int64_t n_probe, uint32_t* counts, uint8_t* build_mark,
                             cudaStream_t st) {
  join_probe_kernel<false><<<grid_for(n_probe, 256, 2), 256, 0, st>>>(K, build_hash, heads, n_buckets - 1, next, probe_hash, probe_ok, n_probe, counts,
                                                                       build_mark, nullptr, nullptr, nullptr);
}
void launch_join_probe_write(const JoinKeys& K, const uint64_t* build_hash, const int32_t* heads, uint64_t n_buckets, const int32_t* next,
                             const uint64_t* probe_hash, const uint8_t* probe_ok, int64_t n_probe, const uint64_t* offsets, int64_t* out_build_idx,
                             int64_t* out_probe_idx, cudaStream_t st) {
  join_probe_kernel<true><<<grid_for(n_probe, 256, 2), 256, 0, st>>>(K, build_hash, heads, n_buckets - 1, next, probe_hash, probe_ok, n_probe, nullptr,
                                                                      nullptr, offsets, out_build_idx, out_probe_idx);
}
__global__ void flag_to_u32_kernel(const uint8_t* flags, uint8_t want, uint32_t* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (flags[i] != 0) == (want != 0);
}
void launch_flag_to_u32(const uint8_t* flags, uint8_t want, uint32_t* out, int64_t n, cudaStream_t st) {
  flag_to_u32_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(flags, want, out, n);
}
__global__ void select_indices_kernel(const uint32_t* flag01, const uint64_t* offs, int64_t* out_idx, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (flag01[i]) out_idx[offs[i]] = i;
}
void launch_select_indices(const uint32_t* flag01, const uint64_t* offs, int64_t* out_idx, int64_t n, cudaStream_t st) {
  select_indices_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(flag01, offs, out_idx, n);
}
__global__ void counts_to_flag_kernel(const uint32_t* counts, uint8_t* flags, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) flags[i] = counts[i] ? 1 : 0;
}
void launch_counts_to_flag(const uint32_t* counts, uint8_t* flags, int64_t n, cudaStream_t st) {
  counts_to_flag_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(counts, flags, n);
}
__global__ void mark_from_idx_kernel(const int64_t* idx, int64_t n, uint8_t* marks) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (idx[i] >= 0) marks[idx[i]] = 1;
}
void launch_mark_from_idx(const int64_t* idx, int64_t n, uint8_t* marks, cudaStream_t st) {
  mark_from_idx_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(idx, n, marks);
}

// ------------------------------------------------------------------------------------------------
// Sort: order-preserving 64-bit key words + stable LSD radix sort of (key, row) pairs
// ------------------------------------------------------------------------------------------------
__global__ void sort_word_kernel(SortWordArgs A, const uint32_t* perm, uint64_t* out, int64_t n) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = perm ? perm[k] : k;
    const bool valid = !A.valid || A.valid[i];
    uint64_t w = 0;
    if (A.word < 0) {  // null-rank word: decides where NULLs go
      w = valid ? (A.nulls_first ? 1 : 0) : (A.nulls_first ? 0 : 1);
      out[k] = w;
      continue;
    }
    if (valid) {
      switch (A.phys) {
        case PH_I8: w = (uint64_t)(int64_t)((const int8_t*)A.data)[i] ^ 0x8000000000000000ull; break;
        case PH_I16: w = (uint64_t)(int64_t)((const int16_t*)A.data)[i] ^ 0x8000000000000000ull; break;
        case PH_I32: w = (uint64_t)(int64_t)((const int32_t*)A.data)[i] ^ 0x8000000000000000ull; break;
        case PH_I64: w = (uint64_t)((const int64_t*)A.data)[i] ^ 0x8000000000000000ull; break;
        case PH_U8:
        case PH_BOOL8: w = ((const uint8_t*)A.data)[i]; break;
        case PH_U16: w = ((const uint16_t*)A.data)[i]; break;
        case PH_U32: w = ((const uint32_t*)A.data)[i]; break;
        case PH_U64: w = ((const uint64_t*)A.data)[i]; break;
        case PH_F32:
        case PH_F64: {
          // raw bits as an INTEGER: if the compiler sees a double here it turns `bits ^ signbit` into an
          // FP negate, and neg.f64 of a NaN does not return the sign-flipped bit pattern (NaN keys were
          // ordered below -0.0); found by tests/test_gpu_sort.py
          long long x = A.phys == PH_F32 ? __double_as_longlong((double)((const float*)A.data)[i]) : ((const long long*)A.data)[i];
          asm volatile("" : "+l"(x));
          x ^= (long long)((unsigned long long)(x >> 63) >> 1);  // IEEE total order
          w = (uint64_t)x ^ 0x8000000000000000ull;
          break;
        }
        case PH_DEC128: {
          const uint64_t* p = (const uint64_t*)A.data + 2 * i;
          w = A.word == 0 ? (p[1] ^ 0x8000000000000000ull) : p[0];  // word 0 = high (signed), word 1 = low
          break;
        }
        case PH_STRVIEW: {
          const unsigned long long* v = (const unsigned long long*)A.data + 2 * i;
          const uint8_t* s = (const uint8_t*)v[0];
          uint32_t len = (uint32_t)v[1];
          uint32_t base = (uint32_t)A.word * 7;  // 7 data bytes per word + 1 "has more/len" byte keeps prefixes ordered
          for (int b = 0; b < 7; b++) {
            uint32_t p = base + b;
            w = (w << 8) | (p < len ? s[p] : 0);
          }
          uint32_t rem = len > base ? len - base : 0;
          w = (w << 8) | (rem > 7 ? 8 : rem);  // bytes present in this word (8 = continues)
          break;
        }
        default: break;
      }
      if (!A.asc) w = ~w;
    }
    out[k] = w;
  }
}
void launch_sort_word(const SortWordArgs& A, const uint32_t* perm, uint64_t* out, int64_t n, cudaStream_t st) {
  sort_word_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(A, perm, out, n);
}
// ---- small-n comparison sort ---------------------------------------------------------------------
// three-way compare of rows i and j under one key; mirrors the word encoding of sort_word_kernel
__device__ __forceinline__ int small_sort_cmp(const SortWordArgs& A, int64_t i, int64_t j) {
  const bool vi = !A.valid || A.valid[i], vj = !A.valid || A.valid[j];
  if (vi != vj) {  // the null-rank word is not affected by asc/desc
    const int ri = vi ? (A.nulls_first ? 1 : 0) : (A.nulls_first ? 0 : 1);
    const int rj = vj ? (A.nulls_first ? 1 : 0) : (A.nulls_first ? 0 : 1);
    return ri < rj ? -1 : 1;
  }
  if (!vi) return 0;
  int c = 0;
  switch (A.phys) {
    case PH_I8: { const int8_t a = ((const int8_t*)A.data)[i], b = ((const int8_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_I16: { const int16_t a = ((const int16_t*)A.data)[i], b = ((const int16_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_I32: { const int32_t a = ((const int32_t*)A.data)[i], b = ((const int32_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_I64: { const int64_t a = ((const int64_t*)A.data)[i], b = ((const int64_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_U8:
    case PH_BOOL8: { const uint8_t a = ((const uint8_t*)A.data)[i], b = ((const uint8_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_U16: { const uint16_t a = ((const uint16_t*)A.data)[i], b = ((const uint16_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_U32: { const uint32_t a = ((const uint32_t*)A.data)[i], b = ((const uint32_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_U64: { const uint64_t a = ((const uint64_t*)A.data)[i], b = ((const uint64_t*)A.data)[j]; c = a < b ? -1 : a > b; break; }
    case PH_F32:
    case PH_F64: {
      long long a = A.phys == PH_F32 ? __double_as_longlong((double)((const float*)A.data)[i]) : ((const long long*)A.data)[i];
      long long b = A.phys == PH_F32 ? __double_as_longlong((double)((const float*)A.data)[j]) : ((const long long*)A.data)[j];
      asm volatile("" : "+l"(a), "+l"(b));  // keep the bit patterns integers (see sort_word_kernel)
      a ^= (long long)((unsigned long long)(a >> 63) >> 1);  // IEEE total order
      b ^= (long long)((unsigned long long)(b >> 63) >> 1);
      c = a < b ? -1 : a > b;
      break;
    }
    case PH_DEC128: {
      const uint64_t* pa = (const uint64_t*)A.data + 2 * i;
      const uint64_t* pb = (const uint64_t*)A.data + 2 * j;
      const int64_t ha = (int64_t)pa[1], hb = (int64_t)pb[1];
      c = ha != hb ? (ha < hb ? -1 : 1) : (pa[0] < pb[0] ? -1 : pa[0] > pb[0]);
      break;
    }
    case PH_STRVIEW: {
      const unsigned long long* va = (const unsigned long long*)A.data + 2 * i;
      const unsigned long long* vb = (const unsigned long long*)A.data + 2 * j;
      const uint8_t* sa = (const uint8_t*)va[0];
      const uint8_t* sb = (const uint8_t*)vb[0];
      const uint32_t la = (uint32_t)va[1], lb = (uint32_t)vb[1], m = la < lb ? la : lb;
      for (uint32_t p = 0; p < m && c == 0; p++) c = sa[p] < sb[p] ? -1 : sa[p] > sb[p];
      if (c == 0) c = la < lb ? -1 : la > lb;
      break;
    }
    default: break;
  }
  return A.asc ? c : -c;
}
__global__ void small_sort_kernel(const SmallSortKeys K, int64_t* perm_out, int64_t n) {
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    int64_t rank = 0;
    for (int64_t j = 0; j < n; j++) {
      int c = 0;
      for (int k = 0; k < K.n_keys && c == 0; k++) c = small_sort_cmp(K.k[k], j, i);
      rank += (c < 0 || (c == 0 && j < i)) ? 1 : 0;  // stable
    }
    perm_out[rank] = i;
  }
}
void launch_small_sort(const SmallSortKeys& K, int64_t* perm_out, int64_t n, cudaStream_t st) {
  if (n <= 0) return;
  small_sort_kernel<<<1, 256, 0, st>>>(K, perm_out, n);
}

__global__ void max_view_len_kernel(const unsigned long long* views, const uint8_t* valid, int64_t n, unsigned int* out_max) {
  unsigned int m = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (!valid || valid[i]) m = max(m, (unsigned int)views[2 * i + 1]);
  m = __reduce_max_sync(0xFFFFFFFFu, m);
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out_max, m);
}
void launch_max_view_len(const unsigned long long* views, const uint8_t* valid, int64_t n, unsigned int* out_max, cudaStream_t st) {
  max_view_len_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(views, valid, n, out_max);
}

static const int RS_BLOCK = 256, RS_ROUNDS = 8, RS_TILE = RS_BLOCK * RS_ROUNDS;

// hist layout: [digit][block] so that one exclusive scan yields global scatter offsets
__global__ void radix_hist_kernel(const uint64_t* keys, int64_t n, int shift, uint32_t* hist, uint32_t n_blocks) {
  __shared__ unsigned int sh[256];
  sh[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int r = 0; r < RS_ROUNDS; r++) {
    int64_t i = base + (int64_t)r * RS_BLOCK + threadIdx.x;
    if (i < n) atomicAdd(&sh[(keys[i] >> shift) & 255], 1u);
  }
  __syncthreads();
  hist[(uint64_t)threadIdx.x * n_blocks + blockIdx.x] = sh[threadIdx.x];
}
__global__ void radix_scatter_kernel(const uint64_t* keys, const uint32_t* vals, uint64_t* keys_out, uint32_t* vals_out, int64_t n, int shift,
                                     const uint64_t* offsets, uint32_t n_blocks) {
  __shared__ unsigned int warp_cnt[8][256];
  __shared__ unsigned long long digit_base[256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  digit_base[threadIdx.x] = offsets[(uint64_t)threadIdx.x * n_blocks + blockIdx.x];
  for (int w = 0; w < 8; w++) warp_cnt[w][threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int r = 0; r < RS_ROUNDS; r++) {
    int64_t i = base + (int64_t)r * RS_BLOCK + threadIdx.x;
    bool ok = i < n;
    uint64_t k = ok ? keys[i] : 0;
    uint32_t v = ok ? vals[i] : 0;
    uint32_t d = ok ? (uint32_t)((k >> shift) & 255) : 0xFFFFFFFFu;
    uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
    uint32_t rank_in_warp = __popc(peers & ((1u << lane) - 1));
    if (ok && rank_in_warp == 0) warp_cnt[warp][d] = __popc(peers);
    __syncthreads();
    if (ok) {
      unsigned long long pos = digit_base[d] + rank_in_warp;
      for (int w = 0; w < warp; w++) pos += warp_cnt[w][d];
      keys_out[pos] = k;
      vals_out[pos] = v;
    }
    __syncthreads();
    {
      unsigned int tot = 0;
      for (int w = 0; w < 8; w++) {
        tot += warp_cnt[w][threadIdx.x];
        warp_cnt[w][threadIdx.x] = 0;
      }
      digit_base[threadIdx.x] += tot;
    }
    __syncthreads();
  }
}
__global__ void radix_skip_check_kernel(const uint32_t* hist, uint32_t n_blocks, int64_t n, unsigned int* skip) {
  // skip the pass if one digit owns every element
  __shared__ unsigned long long tot[256];
  unsigned long long t = 0;
  for (uint32_t b = 0; b < n_blocks; b++) t += hist[(uint64_t)threadIdx.x * n_blocks + b];
  tot[threadIdx.x] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int s = 0;
    for (int d = 0; d < 256; d++)
      if (tot[d] == (unsigned long long)n) s = 1;
    *skip = s;
  }
}

// Small inputs (the tiny ORDER BY stages of TPC-H): one launch, stable rank sort, O(n^2) compares.
__global__ void rank_sort_kernel(const uint64_t* keys, const uint32_t* vals, uint64_t* keys_out, uint32_t* vals_out, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint64_t k = keys[i];
    int rank = 0;
    for (int j = 0; j < n; j++) {
      const uint64_t kj = keys[j];
      rank += (kj < k || (kj == k && j < i)) ? 1 : 0;
    }
    keys_out[rank] = k;
    vals_out[rank] = vals[i];
  }
}

void radix_sort_pairs_u64(uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b, uint32_t* vals_b, int64_t n, uint32_t* hist_scratch,
                          uint64_t* scan_scratch, cudaStream_t st, bool* result_in_a, uint64_t* launches) {
  // hist_scratch: 256*n_blocks u32 ; scan_scratch: 256*n_blocks+1 u64 offsets + scan temp
  if (n <= 4096) {
    rank_sort_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(keys_a, vals_a, keys_b, vals_b, (int)n);
    if (launches) *launches += 1;
    *result_in_a = false;
    return;
  }
  uint32_t n_blocks = (uint32_t)((n + RS_TILE - 1) / RS_TILE);
  if (n_blocks < 1) n_blocks = 1;
  uint64_t* offsets = scan_scratch;
  uint64_t* scan_tmp = scan_scratch + (uint64_t)256 * n_blocks + 1;
  bool in_a = true;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = pass * 8;
    uint64_t* kin = in_a ? keys_a : keys_b;
    uint32_t* vin = in_a ? vals_a : vals_b;
    uint64_t* kout = in_a ? keys_b : keys_a;
    uint32_t* vout = in_a ? vals_b : vals_a;
    radix_hist_kernel<<<n_blocks, RS_BLOCK, 0, st>>>(kin, n, shift, hist_scratch, n_blocks);
    launch_scan_u32_to_u64(hist_scratch, offsets, (int64_t)256 * n_blocks, scan_tmp, st);
    radix_scatter_kernel<<<n_blocks, RS_BLOCK, 0, st>>>(kin, vin, kout, vout, n, shift, offsets, n_blocks);
    if (launches) *launches += 5;
    in_a = !in_a;
  }
  *result_in_a = in_a;
}

// ---- stable partition placement --------------------------------------------------------------------
// dest[i] = (rows of lower partitions) + (earlier rows of the same partition): the reference's
// BatchPartitioner keeps the input order inside every output partition (take() with ascending indices),
// so do we -- stored partitions are then bit-identical from run to run.
__global__ void partition_dest_small_kernel(const uint32_t* ids, int n, uint32_t* dest) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t p = ids[i];
    uint32_t r = 0;
    for (int j = 0; j < n; j++) {
      const uint32_t q = ids[j];
      r += (q < p || (q == p && j < i)) ? 1u : 0u;
    }
    dest[i] = r;
  }
}
__global__ void partition_keys_kernel(const uint32_t* ids, int64_t n, uint64_t* keys, uint32_t* vals) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = ids[i];
    vals[i] = (uint32_t)i;
  }
}
__global__ void invert_perm_kernel(const uint32_t* perm, int64_t n, uint32_t* dest) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) dest[perm[k]] = (uint32_t)k;
}
uint64_t launch_partition_dest_stable(const uint32_t* ids, int64_t n, uint32_t n_bins, uint32_t* dest, uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b,
                                      uint32_t* vals_b, uint32_t* hist_scratch, uint64_t* scan_scratch, cudaStream_t st) {
  if (n <= 0) return 0;
  if (n <= 4096) {
    partition_dest_small_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ids, (int)n, dest);
    return 1;
  }
  partition_keys_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(ids, n, keys_a, vals_a);
  uint64_t launches = 1;
  const int passes = n_bins <= 256 ? 1 : n_bins <= 65536 ? 2 : 4;
  uint32_t n_blocks = (uint32_t)((n + RS_TILE - 1) / RS_TILE);
  uint64_t* offsets = scan_scratch;
  uint64_t* scan_tmp = scan_scratch + (uint64_t)256 * n_blocks + 1;
  bool in_a = true;
  for (int pass = 0; pass < passes; pass++) {
    uint64_t* kin = in_a ? keys_a : keys_b;
    uint32_t* vin = in_a ? vals_a : vals_b;
    uint64_t* kout = in_a ? keys_b : keys_a;
    uint32_t* vout = in_a ? vals_b : vals_a;
    radix_hist_kernel<<<n_blocks, RS_BLOCK, 0, st>>>(kin, n, pass * 8, hist_scratch, n_blocks);
    launch_scan_u32_to_u64(hist_scratch, offsets, (int64_t)256 * n_blocks, scan_tmp, st);
    radix_scatter_kernel<<<n_blocks, RS_BLOCK, 0, st>>>(kin, vin, kout, vout, n, pass * 8, offsets, n_blocks);
    launches += 5;
    in_a = !in_a;
  }
  invert_perm_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(in_a ? vals_a : vals_b, n, dest);
  return launches + 1;
}

// ------------------------------------------------------------------------------------------------
// Synthetic TPC-H input, generated in place in HBM (identical bytes to the host generator)
// ------------------------------------------------------------------------------------------------
__global__ void tpch_fixed_kernel(int table, int col, int kind, int64_t msf, int64_t row0, int64_t n, void* out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t v = tpch::gen_i64(table, col, row0 + i, msf);
    switch (kind) {
      case tpch::K_I64: ((int64_t*)out)[i] = v; break;
      case tpch::K_I32:
      case tpch::K_DATE: ((int32_t*)out)[i] = (int32_t)v; break;
      default: ((ulonglong2*)out)[i] = make_ulonglong2((unsigned long long)v, (unsigned long long)(v >> 63)); break;
    }
  }
}
void launch_tpch_fixed(int table, int col, int kind, int64_t msf, int64_t row0, int64_t n, void* out, cudaStream_t st) {
  tpch_fixed_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(table, col, kind, msf, row0, n, out);
}
__global__ void tpch_str_len_kernel(int table, int col, int64_t msf, int64_t row0, int64_t n, uint32_t* lens) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    char buf[tpch::kMaxStrLen];
    lens[i] = tpch::gen_str(table, col, row0 + i, msf, buf);
  }
}
void launch_tpch_str_len(int table, int col, int64_t msf, int64_t row0, int64_t n, uint32_t* lens, cudaStream_t st) {
  tpch_str_len_kernel<<<grid_for(n, 256, 4), 256, 0, st>>>(table, col, msf, row0, n, lens);
}
__global__ void tpch_str_fill_kernel(int table, int col, int64_t msf, int64_t row0, int64_t n, const uint64_t* offs64, int32_t* offsets, uint8_t* chars) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
    offsets[i] = (int32_t)offs64[i];
    if (i == n) break;
    char buf[tpch::kMaxStrLen];
    uint32_t len = tpch::gen_str(table, col, row0 + i, msf, buf);
    uint8_t* d = chars + offs64[i];
    for (uint32_t k = 0; k < len; k++) d[k] = (uint8_t)buf[k];
  }
}
void launch_tpch_str_fill(int table, int col, int64_t msf, int64_t row0, int64_t n, const uint64_t* offs64, int32_t* offsets, uint8_t* chars,
                          cudaStream_t st) {
  tpch_str_fill_kernel<<<grid_for(n + 1, 256, 2), 256, 0, st>>>(table, col, msf, row0, n, offs64, offsets, chars);
}

}  // namespace b200
