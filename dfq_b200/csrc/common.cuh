// Shared device/host helpers for libdfq_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>

#include "../../include/dfq_b200.h"

namespace dfq {

// ------------------------------------------------------------------------------------------
// host-side error plumbing
// ------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DFQ_CUDA(call)                                                     \
  do {                                                                     \
    cudaError_t _e = (call);                                               \
    if (_e != cudaSuccess) return ::dfq::cuda_fail(_e, #call);             \
  } while (0)

#define DFQ_REQUIRE(cond, msg)                                             \
  do {                                                                     \
    if (!(cond)) {                                                         \
      ::dfq::set_error("%s (%s)", msg, #cond);                             \
      return DFQ_E_ARG;                                                    \
    }                                                                      \
  } while (0)

// Stream-ordered device copy of a small host table; freed with free_async on the same stream.
template <typename T>
int upload(const T* host, int64_t n, T** dev, cudaStream_t st) {
  *dev = nullptr;
  if (n <= 0) return 0;
  DFQ_CUDA(cudaMallocAsync((void**)dev, sizeof(T) * n, st));
  DFQ_CUDA(cudaMemcpyAsync(*dev, host, sizeof(T) * n, cudaMemcpyHostToDevice, st));
  return 0;
}
inline void free_async(void* p, cudaStream_t st) {
  if (p) cudaFreeAsync(p, st);
}

int sm_count();

// All descriptor tables of one call are packed into a MAPPED page-locked staging slot (ring of 4, reused after the copy
// that read it has completed) and moved into ONE stream-ordered device allocation by a small KERNEL that reads the slot over
// PCIe - not by cudaMemcpyAsync: a copy of a few KB queues on the H2D copy engine behind whatever bulk copy is running, and
// in the pipelined host-streaming use (300 MB chunks each way) every launch's tables waited ~6 ms for the NEXT chunk's
// upload to finish, which in turn kept the host from enqueueing the chunk after that (bench.py e2e: 41.7 of 47 GB/s).
// DFQ_TABLES_COPY_ENGINE=1 restores the memcpy path.
struct TablePack {
  struct Item { const void* src; size_t bytes; size_t off; };
  Item items[12];
  int n = 0;
  size_t total = 0;
  unsigned char* dev = nullptr;
  template <typename T>
  int add(const T* host, int64_t count) {       // returns the item index
    const size_t bytes = sizeof(T) * (size_t)(count > 0 ? count : 0);
    items[n] = Item{host, bytes, total};
    total += (bytes + 255) & ~(size_t)255;
    return n++;
  }
  template <typename T>
  T* ptr(int i) const { return (T*)(dev + items[i].off); }
  int upload(cudaStream_t st);                   // 0 or an error code (message set)
  void release(cudaStream_t st) { if (dev) cudaFreeAsync(dev, st); dev = nullptr; }
};

// Small device -> host read-back that stays off the copy engines, like the descriptor upload above: a kernel stores the
// blocks into mapped page-locked memory; the caller synchronizes the stream and copies them out.
struct ReadBack {
  struct Item { void* host; const void* dev; size_t bytes; size_t off; };
  Item items[4];
  int n = 0;
  size_t total = 0;
  int slot = -1;
  unsigned char* mapped = nullptr;
  void add(void* host, const void* dev, size_t bytes) {
    items[n++] = Item{host, dev, bytes, total};
    total += (bytes + 255) & ~(size_t)255;
  }
  int enqueue(cudaStream_t st);   // 0 or an error code (message set)
  void finish();                  // after the stream has been synchronized
  void abandon();                 // error paths: give the slot back without copying
  ~ReadBack() { abandon(); }
};

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
#define DFQ_INF __int_as_float(0x7f800000)

// 128-bit global accesses.  Weights are read once and written once per pass, and inside the
// persistent kernels they are re-read in a later phase after OTHER SMs rewrote them: every access to
// mutable arena data therefore bypasses the (non-coherent) L1 with .cg and is served by L2.
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void stg_stream(float4* p, const float4& v) {
  asm volatile("st.global.cg.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float ldg_stream1(const float* p) {
  float r;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(r) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void stg_stream1(float* p, float v) {
  asm volatile("st.global.cg.f32 [%0], %1;" :: "l"(p), "f"(v) : "memory");
}

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// float atomic min/max through the integer ordering of IEEE bit patterns (works in global and shared).  The branch tests the
// SIGN BIT, not v >= 0: -0.0 (0x80000000) must take the unsigned path of the negatives, where it orders just below +0.0 and
// above every negative number as fminf/fmaxf do; as a signed int it would be INT_MIN, below -inf.
__device__ __forceinline__ void atomic_min_f(float* addr, float v) {
  if (__float_as_int(v) >= 0) atomicMin((int*)addr, __float_as_int(v));
  else                        atomicMax((unsigned int*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* addr, float v) {
  if (__float_as_int(v) >= 0) atomicMax((int*)addr, __float_as_int(v));
  else                        atomicMin((unsigned int*)addr, __float_as_uint(v));
}

// ------------------------------------------------------------------------------------------
// blocked tile partition: the tiles of a phase are numbered consecutively over its task list
// (ptr[q] = first tile of task q, ptr[n] = total); CTA b owns the contiguous range
// [b*T/G, (b+1)*T/G).  A CTA therefore touches only the few tasks its range intersects.
// ------------------------------------------------------------------------------------------
struct TileSpan {
  long long lo, hi;   // global tile range of this CTA
  int q;              // first task intersecting it
};
__device__ __forceinline__ TileSpan tile_span(const long long* __restrict__ ptr, int q_begin, int q_end) {
  TileSpan s;
  const long long first = ptr[q_begin], total = ptr[q_end] - first;
  s.lo = first + (long long)blockIdx.x * total / gridDim.x;
  s.hi = first + (long long)(blockIdx.x + 1) * total / gridDim.x;
  int a = q_begin, b = q_end;   // largest q in [q_begin, q_end) with ptr[q] <= lo
  while (b - a > 1) {
    const int m = (a + b) >> 1;
    if (ptr[m] <= s.lo) a = m; else b = m;
  }
  s.q = a;
  return s;
}

// Block-cyclic walk over the tiles [first, end) of a phase: CTA b visits blocks j*G + b (j = 0, 1, ...) of kTileBlock
// consecutive tiles.  Compared with one contiguous span per CTA this keeps the set of pages all CTAs touch at any time
// within G*kTileBlock tiles (TLB reach; measured: the contiguous split loses 30 % at a 39 GB arena), while a CTA still
// stays on one layer for kTileBlock tiles.
#ifndef DFQ_TILE_BLOCK
#define DFQ_TILE_BLOCK 64
#endif
constexpr long long kTileBlock = DFQ_TILE_BLOCK;

struct TileCursor {
  long long first, end;     // tiles of the phase
  long long t, blk_end;     // current tile, end of the current block
  long long B;              // tiles per block: kTileBlock for a large phase, down to 1 so that a small phase still reaches every CTA
  __device__ __forceinline__ void seek(long long tmin) {   // first tile >= tmin owned by this CTA
    const long long G = gridDim.x, b = blockIdx.x;
    if (tmin < first) tmin = first;
    const long long blk = (tmin - first) / B;
    const long long j = blk / G, r = blk % G;
    long long start_blk;
    if (r == b) { t = tmin; blk_end = first + (blk + 1) * B; return; }
    start_blk = (r < b) ? j * G + b : (j + 1) * G + b;
    t = first + start_blk * B;
    blk_end = t + B;
  }
  __device__ __forceinline__ void init(long long first_, long long end_) {
    first = first_; end = end_;
    const long long per_cta = (end_ - first_) / ((long long)gridDim.x * 4);
    B = per_cta < 1 ? 1 : (per_cta > kTileBlock ? kTileBlock : per_cta);
    seek(first_);
  }
  __device__ __forceinline__ bool valid() const { return t < end; }
  __device__ __forceinline__ void next() {
    if (++t == blk_end) { t += (long long)(gridDim.x - 1) * B; blk_end = t + B; }
  }
};
// largest q in [q_begin, q_end) with ptr[q] <= t
__device__ __forceinline__ int find_task(const long long* __restrict__ ptr, int q_begin, int q_end, long long t) {
  int a = q_begin, b = q_end;
  while (b - a > 1) {
    const int m = (a + b) >> 1;
    if (ptr[m] <= t) a = m; else b = m;
  }
  return a;
}

__device__ __forceinline__ float ld_volatile_f(const float* p) {
  return *(const volatile float*)p;
}

// Scalar prologue of UniformQuantize.forward (utils/quantize.py:49-66) in double, as Python does it.
struct QuantScalars {
  float neg_min;   // fp32(-min_value)       operand of add_(-min_value)
  float min_v;     // fp32(min_value)        operand of the final add_(min_value)
  float scale;     // fp32(scale)            operand of div_/mul_
  float inv_scale; // fp32(1.0 / double scale): reciprocal-multiply mode.  PyTorch CUDA eager computes x.div_(python_float)
                   // as x * float(1.0 / scale) with the reciprocal formed in DOUBLE from the Python scalar [probed on B200
                   // with torch 2.11: 0 mismatches in 4M elements for five scales; float(1.0f / float(scale)) mismatches]
  float qmin, qmax;
};
__host__ __device__ inline QuantScalars quant_scalars(double mn, double mx, int num_bits, int symmetric) {
  QuantScalars q;
  double qmin, qmax, scale;
  if (symmetric) {
    qmin = -ldexp(1.0, num_bits - 1);
    qmax = ldexp(1.0, num_bits - 1) - 1.0;
    mx = fabs(mx);
    mn = fabs(mn);
    if (mx < mn) mx = mn;
    scale = mx / qmax;
    mn = 0.0;
  } else {
    qmin = 0.0;
    qmax = ldexp(1.0, num_bits) - 1.0;
    scale = (mx - mn) / (qmax - qmin);
  }
  // Python max(scale, 1e-8): 1e-8 only if 1e-8 > scale (a NaN scale stays NaN)
  if (1e-8 > scale) scale = 1e-8;
  q.neg_min = (float)(-mn);
  q.min_v = (float)mn;
  q.scale = (float)scale;
  q.inv_scale = (float)(1.0 / scale);
  q.qmin = (float)qmin;
  q.qmax = (float)qmax;
  return q;
}

// quantize.py:70-74, one element.  Every op is individually rounded (no FMA contraction).
template <bool RECIP>
__device__ __forceinline__ float fake_quant(float x, const QuantScalars& q, float* code = nullptr) {
  float t = __fadd_rn(x, q.neg_min);
  t = RECIP ? __fmul_rn(t, q.inv_scale) : __fdiv_rn(t, q.scale);
  t = fminf(fmaxf(t, q.qmin), q.qmax);
  t = rintf(t);
  if (code) *code = t;
  t = __fmul_rn(t, q.scale);
  return __fadd_rn(t, q.min_v);
}

}  // namespace dfq
