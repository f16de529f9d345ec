// Device-side helpers shared by the sm_100a kernels: mbarrier + 1-D bulk (TMA-engine) copies,
// warp-level HMMA, programmatic dependent launch, cache-hinted vector loads.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

constexpr int kWarp = 32;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// 1-D bulk copy global -> shared through the TMA engine (SASS: UBLKCP); completion is signalled
// on `bar` as transaction bytes.  src, dst and bytes must be multiples of 16.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// The same copy with an L2 cache-policy operand.  Weights and K/V tiles are read exactly once per decode step: with the
// evict_first policy the 3.5 GB they add up to stop pushing everything else (kernel instructions, activation vectors,
// norm weights, scales) out of the 126 MB L2 between two uses.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}

// L2 prefetch of a contiguous global range (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void l2_prefetch(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// L2 prefetch of the head of the NEXT kernel's weight stream.  n_tiles > 0: the next GEMV (grid next_grid) gives CTA r
// the contiguous tiles [n_tiles*r/next_grid, n_tiles*(r+1)/next_grid); the first `window` bytes of every region are
// prefetched, one region per calling CTA.  n_tiles == 0: [0, total) as one range, split over the calling CTAs.
// The loops stay rolled: one thread runs them once per launch, and unrolled copies only take instruction-cache space from
// the warps that share the SM.
__device__ __forceinline__ void prefetch_next_stream(const uint8_t* base, int total, int n_tiles, int next_grid,
                                                     int window, int cta, int n_cta) {
  constexpr uint32_t piece = 16384;
  if (n_tiles > 0 && next_grid > 0) {
    const int tile_bytes = total / n_tiles;
#pragma unroll 1
    for (int r = cta; r < next_grid; r += n_cta) {
      const long long t0 = ((long long)n_tiles * r) / next_grid, t1 = ((long long)n_tiles * (r + 1)) / next_grid;
      const long long bytes = min((t1 - t0) * (long long)tile_bytes, (long long)window);
      const uint8_t* src = base + t0 * tile_bytes;
#pragma unroll 1
      for (long long off = 0; off < bytes; off += piece)
        l2_prefetch(src + off, (uint32_t)min((long long)piece, bytes - off) & ~15u);
    }
  } else {
    const int n_piece = (total + (int)piece - 1) / (int)piece;
#pragma unroll 1
    for (int i = cta; i < n_piece; i += n_cta) {
      const uint32_t off = (uint32_t)i * piece;
      const uint32_t len = min(piece, (uint32_t)total - off) & ~15u;
      if (len) l2_prefetch(base + off, len);
    }
  }
}

// ---- programmatic dependent launch -----------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- named barriers (sub-block sync) ---------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- HMMA m16n8k16 f16 x f16 -> f32 ----------------------------------------------------------
// A (16x16, row): a0:(g, 2t..2t+1) a1:(g+8, 2t..) a2:(g, 2t+8..) a3:(g+8, 2t+8..)
// B (16x8,  col): b0:(k=2t..2t+1, n=g) b1:(k=2t+8.., n=g)
// C (16x8):       c0,c1:(g, 2t..2t+1)  c2,c3:(g+8, 2t..2t+1)         g = lane/4, t = lane%4
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                         uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ---- loads -----------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
// L2-coherent 16-byte load (ld.global.cg): never served from a stale L1 line when another CTA of the SAME launch wrote
// the data (persistent kernels with grid barriers)
__device__ __forceinline__ uint4 ldg_cg_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
// Loads that ask the L2 to keep the line (evict_last priority): small per-layer constants (norm weights, scales) are read
// once per decode step, 3.5 GB of streamed weights apart; without the hint every read is an HBM miss that queues behind
// the weight stream of the kernel that needs it (measured: x staging of the QKV launch waited ~5 us for its norm weight).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint4 ldg_keep_v4(const void* p, uint64_t pol) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ uint32_t ldg_keep_u32(const void* p, uint64_t pol) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ uint4 lds_v4(const void* p) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "r"(smem_u32(p)));
  return r;
}
__device__ __forceinline__ uint2 lds_v2(const void* p) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(smem_u32(p)));
  return r;
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ---- optional per-launch timeline (B200 %globaltimer, ns): [0]=first CTA start (min), [1]=x staged (max),
// [2]=last MMA warp done (max), [3]=last CTA end (max).  tl == nullptr -> off.
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void tl_min(unsigned long long* tl, int i) {
  if (tl) atomicMin(tl + i, gtime_ns());
}
__device__ __forceinline__ void tl_max(unsigned long long* tl, int i) {
  if (tl) atomicMax(tl + i, gtime_ns());
}

// per-CTA stamps of selected launches (b200_timeline_cta): row = CTA, 16 columns (0..7 as in the timeline row, 8.. = finer stamps)
__device__ __forceinline__ void tl_cta(unsigned long long* tlc, int cta, int i) {
  if (tlc) tlc[(size_t)cta * 16 + i] = gtime_ns();
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

}  // namespace b200
