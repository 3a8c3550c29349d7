// Kernel (1): CSR gather + weighted sum + L2 normalise -- the class-bank builder.
//
//   out[r] = normalize( sum_{j in CSR row row_map[r]} w[j] * E[col[j]] )      (fp32 math)
//
// Reference: update_classifier's `text_feats / text_feats.norm(dim=-1, keepdim=True)`
// (model/clip_tree.py:323) is the identity-CSR case; the image-feature normalisation of
// forward (model/clip_tree.py:330) uses the same kernel.  The multi-node rows implement the
// hierarchy aggregation of north_star (operator shape: baseline/DGP/models/gcn_dense_att.py).
//
// HBM-bound: one warp per output row, 128-bit read-only loads that bypass L1 (each source row
// is streamed once per gather), fp32 accumulators in registers, warp-shuffle reduction of the
// squared norm, one 128-bit store per lane and vector.  Compulsory traffic per row:
// nnz_row * D * sizeof(in) + D * sizeof(out) (+ CSR).
#include "placement.cuh"

namespace hgr {
namespace {

__device__ __forceinline__ uint4 ldg_nc_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

template <typename T>
struct Vec8;  // 8 consecutive elements <-> float[8]

template <>
struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* p, float (&f)[8]) {
    // a lane's 32 bytes are one sector read by two 16-byte loads: keep the line in L1
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
    f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&f)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
  }
};

template <>
struct Vec8<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    uint4 a = ldg_nc_u4(p);
    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift
      f[2 * i] = __uint_as_float(u[i] << 16);
      f[2 * i + 1] = __uint_as_float(u[i] & 0xFFFF0000u);
    }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    uint4 o;
    uint32_t* u = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      u[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = o;
  }
};

template <>
struct Vec8<__half> {
  static __device__ __forceinline__ void load(const __half* p, float (&f)[8]) {
    uint4 a = ldg_nc_u4(p);
    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 t = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// MAXV = 8-element vectors per lane held in registers (covers D <= 256 * MAXV).
template <typename TIn, typename TOut, int MAXV>
__global__ void __launch_bounds__(256)
aggregate_normalize_kernel(const TIn* __restrict__ E, int D8, const int32_t* __restrict__ rowptr,
                           const int32_t* __restrict__ col, const float* __restrict__ w,
                           const int32_t* __restrict__ row_map, int64_t n_out, TOut* __restrict__ out,
                           float* __restrict__ out_norm) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t D = static_cast<int64_t>(D8) * 8;

  for (int64_t row = warp0; row < n_out; row += nwarps) {
    const int32_t src = row_map ? row_map[row] : static_cast<int32_t>(row);
    int32_t beg = src, end = src + 1;
    if (rowptr) {
      beg = rowptr[src];
      end = rowptr[src + 1];
    }
    float acc[MAXV][8];
#pragma unroll
    for (int v = 0; v < MAXV; ++v)
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[v][e] = 0.f;

    // The row's column ids / weights are fetched by the whole warp in one coalesced load (32 entries at a time)
    // and broadcast by shuffle -- no per-entry dependent scalar load -- and TWO source rows are in flight per step:
    // with ~2 entries per row (ancestor chains) a row costs one gather round trip instead of a chain of them.
    // (Also tried: prefetching the next row's pointers / ids one row ahead -- no gain, the gather itself dominates.)
    const int32_t n = end - beg;
    int32_t myc = src;
    float myw = 1.f;
    for (int32_t j0 = 0; j0 < n; j0 += 2) {
      if ((j0 & 31) == 0 && rowptr) {
        const int32_t j = beg + j0 + lane;
        myc = j < end ? __ldg(col + j) : 0;
        myw = (j < end && w) ? __ldg(w + j) : 1.f;
      }
      const bool two = j0 + 1 < n;
      const int32_t c0 = __shfl_sync(0xffffffffu, myc, j0 & 31);
      const int32_t c1 = __shfl_sync(0xffffffffu, myc, (j0 + 1) & 31);
      const float w0 = __shfl_sync(0xffffffffu, myw, j0 & 31);
      const float w1 = two ? __shfl_sync(0xffffffffu, myw, (j0 + 1) & 31) : 0.f;
      const TIn* s0 = E + static_cast<int64_t>(c0) * D;
      const TIn* s1 = E + static_cast<int64_t>(two ? c1 : c0) * D;
      float f0[MAXV][8], f1[MAXV][8];
#pragma unroll
      for (int v = 0; v < MAXV; ++v) {  // issue all loads of both source rows first
        const int idx = lane + 32 * v;
        if (idx < D8) {
          Vec8<TIn>::load(s0 + idx * 8, f0[v]);
          Vec8<TIn>::load(s1 + idx * 8, f1[v]);
        }
      }
#pragma unroll
      for (int v = 0; v < MAXV; ++v) {
        const int idx = lane + 32 * v;
        if (idx < D8) {
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[v][e] = fmaf(w1, f1[v][e], fmaf(w0, f0[v][e], acc[v][e]));
        }
      }
    }

    float ss = 0.f;
#pragma unroll
    for (int v = 0; v < MAXV; ++v)
#pragma unroll
      for (int e = 0; e < 8; ++e) ss = fmaf(acc[v][e], acc[v][e], ss);
    ss = warp_sum(ss);
    const float nrm = sqrtf(ss);
    if (out_norm && lane == 0) out_norm[row] = nrm;

    TOut* dst = out + row * D;
#pragma unroll
    for (int v = 0; v < MAXV; ++v) {
      const int idx = lane + 32 * v;
      if (idx < D8) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = __fdiv_rn(acc[v][e], nrm);  // x / ||x||, as the reference divides
        Vec8<TOut>::store(dst + idx * 8, o);
      }
    }
  }
}

// Identity CSR (row r = {src}, weight 1): the plain row normalise of update_classifier / forward.  No
// accumulators besides the row itself, one row per warp, 3 CTAs per SM: 24 rows in flight per SM on the 21,841-row
// bank, and at most 72 registers, so that a CTA of it fits on an SM beside a resident scoring CTA and a merge CTA
// (DESIGN.md section 4).  (Two rows per warp in flight took 101-108 registers, and 85 with spills.)
template <typename TIn, typename TOut, int MAXV>
__global__ void __launch_bounds__(256, 3)
normalize_rows_kernel(const TIn* __restrict__ E, int D8, const int32_t* __restrict__ row_map, int64_t n_out,
                      TOut* __restrict__ out, float* __restrict__ out_norm, TOut* __restrict__ out2 = nullptr,
                      const int32_t* __restrict__ dst_map = nullptr) {
  HGR_PLACE_ENTER();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t D = static_cast<int64_t>(D8) * 8;
  for (int64_t row = warp0; row < n_out; row += nwarps) {
    const int64_t src = row_map ? row_map[row] : row;
    float a[MAXV][8];
#pragma unroll
    for (int v = 0; v < MAXV; ++v) {
      const int idx = lane + 32 * v;
      if (idx < D8) {
        Vec8<TIn>::load(E + src * D + idx * 8, a[v]);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) a[v][e] = 0.f;
      }
    }
    float ss = 0.f;
#pragma unroll
    for (int v = 0; v < MAXV; ++v)
#pragma unroll
      for (int e = 0; e < 8; ++e) ss = fmaf(a[v][e], a[v][e], ss);
    ss = warp_sum(ss);
    const float n = sqrtf(ss);
    if (out_norm && lane == 0) out_norm[row] = n;
    // second destination (dual form): row r also lands at row dst_map[r] of out2 -- the test-class bank in its own
    // row order, written by the same pass that writes the all-node bank
    const int64_t d = dst_map ? dst_map[row] : -1;
#pragma unroll
    for (int v = 0; v < MAXV; ++v) {
      const int idx = lane + 32 * v;
      if (idx < D8) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = __fdiv_rn(a[v][e], n);
        Vec8<TOut>::store(out + row * D + idx * 8, o);
        if (d >= 0) Vec8<TOut>::store(out2 + d * D + idx * 8, o);
      }
    }
  }
  HGR_PLACE_LEAVE(kNormalize);
}

// Row normalise with BROADCAST stores: row r of the local block lands at row (row0 + r) of every destination
// (bf16 [*, D] arrays; local or peer memory).  Feature ingest of the class-sharded head: every rank copies only
// its own block of image rows from the host, and the normalised A operand is replicated over NVLink by the
// producing kernel (16-byte stores, 512 contiguous bytes per warp instruction).
struct BcastDst {
  __nv_bfloat16* p[16];
};
template <typename TIn, int MAXV>
__global__ void __launch_bounds__(256)
normalize_bcast_kernel(const TIn* __restrict__ E, int D8, int64_t n_rows, int64_t row0, BcastDst dst, int n_dst) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t D = static_cast<int64_t>(D8) * 8;
  for (int64_t row = warp0; row < n_rows; row += nwarps) {
    float a[MAXV][8];
#pragma unroll
    for (int v = 0; v < MAXV; ++v) {
      const int idx = lane + 32 * v;
      if (idx < D8) {
        Vec8<TIn>::load(E + row * D + idx * 8, a[v]);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) a[v][e] = 0.f;
      }
    }
    float ss = 0.f;
#pragma unroll
    for (int v = 0; v < MAXV; ++v)
#pragma unroll
      for (int e = 0; e < 8; ++e) ss = fmaf(a[v][e], a[v][e], ss);
    ss = warp_sum(ss);
    const float n = sqrtf(ss);
#pragma unroll
    for (int v = 0; v < MAXV; ++v) {
      const int idx = lane + 32 * v;
      if (idx < D8) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = __fdiv_rn(a[v][e], n);
        for (int g = 0; g < n_dst; ++g) Vec8<__nv_bfloat16>::store(dst.p[g] + (row0 + row) * D + idx * 8, o);
      }
    }
  }
}

// Any D (multiple of 8): two passes over the gathered rows, nothing kept in registers.
template <typename TIn, typename TOut>
__global__ void __launch_bounds__(256)
aggregate_normalize_generic_kernel(const TIn* __restrict__ E, int D8, const int32_t* __restrict__ rowptr,
                                   const int32_t* __restrict__ col, const float* __restrict__ w,
                                   const int32_t* __restrict__ row_map, int64_t n_out,
                                   TOut* __restrict__ out, float* __restrict__ out_norm) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t D = static_cast<int64_t>(D8) * 8;
  for (int64_t row = warp0; row < n_out; row += nwarps) {
    const int32_t src = row_map ? row_map[row] : static_cast<int32_t>(row);
    int32_t beg = src, end = src + 1;
    if (rowptr) {
      beg = rowptr[src];
      end = rowptr[src + 1];
    }
    float nrm = 0.f;
    for (int pass = 0; pass < 2; ++pass) {
      float ss = 0.f;
      for (int idx = lane; idx < D8; idx += 32) {
        float a[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = 0.f;
        for (int32_t j = beg; j < end; ++j) {
          const int32_t c = rowptr ? col[j] : j;
          const float wj = (rowptr && w) ? w[j] : 1.f;
          float f[8];
          Vec8<TIn>::load(E + static_cast<int64_t>(c) * D + idx * 8, f);
#pragma unroll
          for (int e = 0; e < 8; ++e) a[e] = fmaf(wj, f[e], a[e]);
        }
        if (pass == 0) {
#pragma unroll
          for (int e = 0; e < 8; ++e) ss = fmaf(a[e], a[e], ss);
        } else {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = __fdiv_rn(a[e], nrm);
          Vec8<TOut>::store(out + row * D + idx * 8, o);
        }
      }
      if (pass == 0) {
        nrm = sqrtf(warp_sum(ss));
        if (out_norm && lane == 0) out_norm[row] = nrm;
      }
    }
  }
}

template <typename TIn, typename TOut>
int dispatch(const void* E, int64_t D, const int32_t* rowptr, const int32_t* col, const float* w,
             const int32_t* row_map, int64_t n_out, void* out, float* out_norm, cudaStream_t stream) {
  const int D8 = static_cast<int>(D / 8);
  const int threads = 256;
  const int64_t rows_per_block = threads / 32;
  int64_t want = (n_out + rows_per_block - 1) / rows_per_block;
  const int64_t cap = static_cast<int64_t>(num_sms()) * 8;  // 8 resident CTAs of 256 threads per SM
  const int blocks = static_cast<int>(want < cap ? (want < 1 ? 1 : want) : cap);
  const TIn* e = static_cast<const TIn*>(E);
  TOut* o = static_cast<TOut*>(out);
  if (rowptr == nullptr && D8 <= 128) {  // identity CSR: the specialised row normalise
    const int64_t capn = static_cast<int64_t>(num_sms()) * 3;   // one wave (launch bounds)
    const int64_t wantn = (n_out + rows_per_block - 1) / rows_per_block;
    const int nb = static_cast<int>(wantn < capn ? (wantn < 1 ? 1 : wantn) : capn);
    if (D8 <= 32) normalize_rows_kernel<TIn, TOut, 1><<<nb, threads, 0, stream>>>(e, D8, row_map, n_out, o, out_norm);
    else if (D8 <= 64) normalize_rows_kernel<TIn, TOut, 2><<<nb, threads, 0, stream>>>(e, D8, row_map, n_out, o, out_norm);
    else if (D8 <= 96) normalize_rows_kernel<TIn, TOut, 3><<<nb, threads, 0, stream>>>(e, D8, row_map, n_out, o, out_norm);
    else normalize_rows_kernel<TIn, TOut, 4><<<nb, threads, 0, stream>>>(e, D8, row_map, n_out, o, out_norm);
    HGR_CHECK_LAUNCH();
    return HGR_OK;
  }
  // one wave: as many CTAs as are resident at once (register-limited), each warp strides over the rows
#define HGR_AGG_LAUNCH(MAXV)                                                                                      \
  do {                                                                                                            \
    int per_sm = 1;                                                                                               \
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, aggregate_normalize_kernel<TIn, TOut, MAXV>, threads, 0); \
    const int64_t wave = static_cast<int64_t>(num_sms()) * (per_sm < 1 ? 1 : per_sm);                              \
    const int nblk = static_cast<int>(want < wave ? (want < 1 ? 1 : want) : wave);                                \
    aggregate_normalize_kernel<TIn, TOut, MAXV><<<nblk, threads, 0, stream>>>(e, D8, rowptr, col, w, row_map,     \
                                                                              n_out, o, out_norm);                \
  } while (0)
  if (D8 <= 32) HGR_AGG_LAUNCH(1);
  else if (D8 <= 64) HGR_AGG_LAUNCH(2);
  else if (D8 <= 96) HGR_AGG_LAUNCH(3);
  else if (D8 <= 128) HGR_AGG_LAUNCH(4);
  else if (D8 <= 256) HGR_AGG_LAUNCH(8);
  else
    aggregate_normalize_generic_kernel<TIn, TOut><<<blocks, threads, 0, stream>>>(e, D8, rowptr, col, w, row_map,
                                                                                   n_out, o, out_norm);
#undef HGR_AGG_LAUNCH
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace

template <typename TIn>
static int dispatch_bcast(const void* E, int64_t D, int64_t n_rows, int64_t row0, int n_dst, void* const* dst,
                          cudaStream_t stream) {
  BcastDst d{};
  for (int g = 0; g < n_dst; ++g) d.p[g] = static_cast<__nv_bfloat16*>(dst[g]);
  const int D8 = static_cast<int>(D / 8);
  const int64_t want = (n_rows + 7) / 8;
  const int64_t cap = static_cast<int64_t>(num_sms()) * 4;
  const int nb = static_cast<int>(want < cap ? (want < 1 ? 1 : want) : cap);
  const TIn* e = static_cast<const TIn*>(E);
  if (D8 <= 32) normalize_bcast_kernel<TIn, 1><<<nb, 256, 0, stream>>>(e, D8, n_rows, row0, d, n_dst);
  else if (D8 <= 64) normalize_bcast_kernel<TIn, 2><<<nb, 256, 0, stream>>>(e, D8, n_rows, row0, d, n_dst);
  else if (D8 <= 96) normalize_bcast_kernel<TIn, 3><<<nb, 256, 0, stream>>>(e, D8, n_rows, row0, d, n_dst);
  else normalize_bcast_kernel<TIn, 4><<<nb, 256, 0, stream>>>(e, D8, n_rows, row0, d, n_dst);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_normalize_bcast(const void* E, int e_dtype, int64_t n_rows, int64_t D, int64_t row0, int n_dst,
                           void* const* dst, cudaStream_t stream) {
  if (n_rows == 0) return HGR_OK;
  if (D > 1024) return set_error(HGR_ERR_UNSUPPORTED, "hgr_normalize_rows_bcast: D = %lld > 1024", (long long)D);
  if (e_dtype == HGR_F32) return dispatch_bcast<float>(E, D, n_rows, row0, n_dst, dst, stream);
  if (e_dtype == HGR_F16) return dispatch_bcast<__half>(E, D, n_rows, row0, n_dst, dst, stream);
  if (e_dtype == HGR_BF16) return dispatch_bcast<__nv_bfloat16>(E, D, n_rows, row0, n_dst, dst, stream);
  return set_error(HGR_ERR_UNSUPPORTED, "hgr_normalize_rows_bcast: dtype %d not supported", e_dtype);
}

template <typename TIn>
static int dual_dispatch(const void* E, int64_t n_rows, int64_t D, __nv_bfloat16* out, const int32_t* dst_map,
                         __nv_bfloat16* out2, cudaStream_t stream) {
  const int D8 = static_cast<int>(D / 8);
  const int threads = 256;
  const int64_t rows_per_block = threads / 32;
  const int64_t capn = static_cast<int64_t>(num_sms()) * 3;   // one wave (launch bounds)
  const int64_t wantn = (n_rows + rows_per_block - 1) / rows_per_block;
  const int nb = static_cast<int>(wantn < capn ? (wantn < 1 ? 1 : wantn) : capn);
  const TIn* e = static_cast<const TIn*>(E);
  if (D8 <= 32) normalize_rows_kernel<TIn, __nv_bfloat16, 1><<<nb, threads, 0, stream>>>(e, D8, nullptr, n_rows, out, nullptr, out2, dst_map);
  else if (D8 <= 64) normalize_rows_kernel<TIn, __nv_bfloat16, 2><<<nb, threads, 0, stream>>>(e, D8, nullptr, n_rows, out, nullptr, out2, dst_map);
  else if (D8 <= 96) normalize_rows_kernel<TIn, __nv_bfloat16, 3><<<nb, threads, 0, stream>>>(e, D8, nullptr, n_rows, out, nullptr, out2, dst_map);
  else normalize_rows_kernel<TIn, __nv_bfloat16, 4><<<nb, threads, 0, stream>>>(e, D8, nullptr, n_rows, out, nullptr, out2, dst_map);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

template <typename TIn>
static int normalize_footprint_of(int64_t D, int32_t* out) {
  const int D8 = static_cast<int>(D / 8);
  cudaFuncAttributes fa;
  if (D8 <= 32) HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, normalize_rows_kernel<TIn, __nv_bfloat16, 1>));
  else if (D8 <= 64) HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, normalize_rows_kernel<TIn, __nv_bfloat16, 2>));
  else if (D8 <= 96) HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, normalize_rows_kernel<TIn, __nv_bfloat16, 3>));
  else HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, normalize_rows_kernel<TIn, __nv_bfloat16, 4>));
  out[0] = 256;
  out[1] = fa.numRegs;
  out[2] = static_cast<int32_t>(fa.sharedSizeBytes);
  out[3] = 0;
  return HGR_OK;
}

int normalize_rows_footprint(int e_dtype, int64_t D, int32_t* out) {
  if (D < 8 || D % 8 != 0 || D > 1024) return set_error(HGR_ERR_UNSUPPORTED, "normalise footprint: D = %lld", (long long)D);
  if (e_dtype == HGR_F32) return normalize_footprint_of<float>(D, out);
  if (e_dtype == HGR_F16) return normalize_footprint_of<__half>(D, out);
  if (e_dtype == HGR_BF16) return normalize_footprint_of<__nv_bfloat16>(D, out);
  return set_error(HGR_ERR_UNSUPPORTED, "normalise footprint: dtype %d not supported", e_dtype);
}

#ifdef HGR_PLACEMENT
int placement_attach_normalize(const place::Log& l) { return place::attach(l); }
#endif

int launch_normalize_dual(const void* E, int e_dtype, int64_t n_rows, int64_t D, void* out, const int32_t* dst_map,
                          void* out2, cudaStream_t stream) {
  if (D / 8 > 128) return set_error(HGR_ERR_UNSUPPORTED, "hgr_normalize_rows_dual: D = %lld > 1024", (long long)D);
  __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
  __nv_bfloat16* o2 = static_cast<__nv_bfloat16*>(out2);
  if (e_dtype == HGR_F32) return dual_dispatch<float>(E, n_rows, D, o, dst_map, o2, stream);
  if (e_dtype == HGR_BF16) return dual_dispatch<__nv_bfloat16>(E, n_rows, D, o, dst_map, o2, stream);
  if (e_dtype == HGR_F16) return dual_dispatch<__half>(E, n_rows, D, o, dst_map, o2, stream);
  return set_error(HGR_ERR_BAD_ARG, "hgr_normalize_rows_dual: unknown dtype %d", e_dtype);
}

int launch_aggregate_normalize(const void* E, int e_dtype, int64_t n_src, int64_t D, const int32_t* rowptr,
                               const int32_t* col, const float* w, const int32_t* row_map, int64_t n_out,
                               void* out, int out_dtype, float* out_norm, cudaStream_t stream) {
  (void)n_src;
  if (n_out == 0) return HGR_OK;
#define HGR_AGG_CASE(EI, TI, EO, TO) \
  if (e_dtype == EI && out_dtype == EO) return dispatch<TI, TO>(E, D, rowptr, col, w, row_map, n_out, out, out_norm, stream)
  HGR_AGG_CASE(HGR_F32, float, HGR_BF16, __nv_bfloat16);
  HGR_AGG_CASE(HGR_F32, float, HGR_F32, float);
  HGR_AGG_CASE(HGR_BF16, __nv_bfloat16, HGR_BF16, __nv_bfloat16);
  HGR_AGG_CASE(HGR_BF16, __nv_bfloat16, HGR_F32, float);
  HGR_AGG_CASE(HGR_F16, __half, HGR_BF16, __nv_bfloat16);
  HGR_AGG_CASE(HGR_F16, __half, HGR_F32, float);
#undef HGR_AGG_CASE
  return set_error(HGR_ERR_UNSUPPORTED, "hgr_aggregate_normalize: dtype pair (%d -> %d) not supported", e_dtype,
                   out_dtype);
}

}  // namespace hgr
