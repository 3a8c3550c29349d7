// Placement diagnostics, compiled only with -DHGR_PLACEMENT (tools/build_variant.sh; never in the production build).
// The scoring, row-normalise and select-merge kernels log per CTA the SM it ran on and %globaltimer at entry and
// exit, so that tools/placement.py can tell how much of the small kernels' time shared an SM with a scoring CTA.
// The scoring kernel also counts the chunks its deferred-insert epilogue scanned and how many of them found a queue
// too full for the roomy append.  The instrumentation costs registers (ptxas, CUDA 12.9: scoring <4,8> 180 instead of
// 167, normalise <bf16,bf16,4> 75 instead of 68), so the variant's own budget is tighter than production's.
#pragma once
#include "common.cuh"

#ifdef HGR_PLACEMENT
namespace hgr {
namespace place {

enum Kind : uint32_t { kScore = 1, kNormalize = 2, kMerge = 3 };
struct Rec {
  unsigned long long t0, t1;   // %globaltimer (ns) at CTA entry and exit
  uint32_t sm, kind;
};
struct Log {
  Rec* rec;
  unsigned int* n;               // records written (may pass cap: those beyond it are dropped)
  unsigned int cap;
  unsigned long long* chunks;    // [0] chunks scanned by top-K epilogue warps, [1] of them not roomy
};
static __device__ Log g_log;    // one copy per translation unit: placement_attach_* set each

static int attach(const Log& l) {
  HGR_CHECK_CUDA(cudaMemcpyToSymbol(g_log, &l, sizeof(Log)));
  return HGR_OK;
}
__device__ __forceinline__ unsigned long long now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void leave(uint32_t kind, unsigned long long t0) {
  const Log l = g_log;
  if (l.rec == nullptr) return;
  uint32_t sm;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
  const unsigned int i = atomicAdd(l.n, 1u);
  if (i < l.cap) l.rec[i] = Rec{t0, now(), sm, kind};
}
__device__ __forceinline__ void count_chunks(unsigned long long chunks, unsigned long long crowded) {
  const Log l = g_log;
  if (l.chunks == nullptr) return;
  atomicAdd(l.chunks, chunks);
  atomicAdd(l.chunks + 1, crowded);
}

}  // namespace place
int placement_attach_normalize(const place::Log& l);   // aggregate_norm.cu
int placement_attach_merge(const place::Log& l);       // topk_merge.cu
}  // namespace hgr

// at the top of a kernel / at its end, where every thread of the CTA arrives
#define HGR_PLACE_ENTER() const unsigned long long hgr_place_t0 = ::hgr::place::now()
#define HGR_PLACE_LEAVE(kind)                                                  \
  do {                                                                         \
    __syncthreads();                                                           \
    if (threadIdx.x == 0) ::hgr::place::leave(::hgr::place::kind, hgr_place_t0); \
  } while (0)
#else
#define HGR_PLACE_ENTER() \
  do {                    \
  } while (0)
#define HGR_PLACE_LEAVE(kind) \
  do {                        \
  } while (0)
#endif
