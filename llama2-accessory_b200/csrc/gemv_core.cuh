// Shared device code of the GEMV family: constants, parameters, codecs, x staging, epilogue and MMA roles.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <string>

#include "../../include/b200_decode.h"
#include "common.cuh"
#include "ll.cuh"

namespace b200 {
void set_error(const std::string& s);
int sm_count();
size_t smem_optin();
unsigned long long* timeline_slot();
unsigned long long* timeline_cta_slot();
int prefetch_window_bytes();  // B200_PF_KB (default 96) * 1024
int tune_get(const char* name, int dflt);  // b200_tune override, else environment, else default (api.cu)
struct GemvParams;
// validate one b200_gemv_args_t and fill the device parameter block (gemv.cu); returns 0 or a B200_E_* code
int build_gemv_params(const b200_gemv_args_t* a, GemvParams* p);
// bs = 1 integer-path kernel (gemv1.cu): does it cover this call / launch it
bool gemv1_supported(const b200_gemv_args_t* a, const GemvParams& p);
int gemv1_launch(const b200_gemv_args_t* a, GemvParams p, cudaStream_t st);

constexpr int kConsumerWarps = 16;  // MMA warps: 4 per scheduler hide the LDS -> LOP3 -> HMMA latency chain
constexpr int kConsumerThreads = kConsumerWarps * 32;
constexpr int kEpiWarps = 2;
constexpr int kThreads = kConsumerThreads + 32 + kEpiWarps * 32;  // + producer warp + epilogue warps
#ifndef B200_KCHUNK
#define B200_KCHUNK 2
#endif
constexpr int kChunk = B200_KCHUNK;              // k-blocks per warp per ring slot
constexpr int kSlotBlocks = kConsumerWarps * kChunk;
constexpr int kSlotBytes = kSlotBlocks * 512;
constexpr int kXPad = 32;  // halfs of padding per staged x row (64 B: rows g, g+1 hit different banks)
constexpr float kTwo24 = 16777216.0f;
constexpr float kInvTwo24 = 1.0f / 16777216.0f;

struct GemvParams {
  int bits;
  const uint8_t* qw;
  const __half2* sz;
  int N, K, Kpad, n_tiles, KB, G, gb_mask, gb_shift, gs_chunks;
  int T;
  int pro;
  const __half* xin;
  const __half* resid;
  const __half* delta;
  __half* h_out;
  const __half* gamma;
  float eps;
  int epi;
  void* out;
  int n_q_rows, n_kv_rows;
  const float2* rope;
  const int* pos;
  int tokens_per_seq;
  __half* kcache;
  __half* vtcache;
  int cache_seq, hkv;
  const int* slot_expert;
  int expert_id, n_slots, src_div;
  int slot_lo, slot_hi;  // MoE: this launch takes the routed slots of rank [slot_lo, slot_hi) among those of its expert (token-group split)
  int t_base;            // token index of column 0 in the caller's batch (token-group split of a QKV launch)
  int stages, x_stride, n_chunk64;
  const uint8_t* next_w;  // the NEXT kernel's weight stream; region heads are prefetched into L2 by the producer
  int next_bytes, next_tiles, next_grid, next_window;
  int prefetch_kv;  // QKV launch: the producer also pulls the K/V rows the following attention kernel reads into L2
  int stream_ef;               // weight bulk copies carry the L2 evict_first policy (B200_STREAM_EF)
  int keep_const;              // norm weight / scales loaded with the L2 evict_last hint (B200_KEEP_CONST)
  const uint8_t* const_pf;     // a later kernel's small constants (its norm weight): CTA 0 prefetches them into L2 first thing
  int const_pf_bytes;
  // tensor parallelism inside the persistent kernel (mega1.cu): `delta` is n_delta rank partials [n_delta][K] summed in
  // rank order (fp32, one rounding -- the all-reduce of a RowParallelLinear, quant.py:41), and the epilogue stores its
  // rows into the n_bcast peer buffers bcast[r] (+ bcast_off elements) instead of `out`
  int n_delta, n_bcast, bcast_off;
  void* bcast[8];
  // stand-alone kernels at TP > 1 (bs = 1): the same data movement in the flag-in-data format of ll.cuh, so that NO
  // collective runs between the kernels.  ll_out: the epilogue stores {half2, seq} units into bcast[r] (peer-mapped);
  // ll_in: `delta` is an LL buffer [n_delta][K/2 units].  seq = *ll_step * ll_period + id + 1 (ll_step: device counter
  // of decode steps, advanced once per step by the caller).
  int ll_out, ll_in, ll_out_id, ll_in_id, ll_period;
  const unsigned* ll_step;
  unsigned* ll_err;
  unsigned long long* tl;  // optional timeline row
  unsigned long long* tlc;  // optional per-CTA stamps [grid][8] (b200_timeline_cta)
  int dbg;  // experiment knob (B200_GEMV_DBG): 1 = skip the MMA math, 2 = skip the weight LDS too
};

// ------------------------------------------------------------------------------------------------
// Codecs: one packed 512-byte k-block (uint4 per lane) -> HMMAs.  acc[nt][cls][4].
// xr[nt] points at the lane's k-run of the staged x row for n-tile nt (block offset added here).
// ------------------------------------------------------------------------------------------------
template <int BITS>
struct Codec;

// 32-bit shared-memory loads (addresses precomputed once per warp: no cvta / 64-bit math in the hot loop)
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a));
  return r;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(a));
  return r;
}

// Every codec exposes  XF (the lane's B fragments of one k-block), load_x(addr, XF&), math(w, XF, acc[NCLS][4]).
template <>
struct Codec<4> {
  static constexpr int KBLK = 64, NCLS = 2, LANE_K = 16;
  struct XF { uint4 a, b; };
  static __device__ __forceinline__ void load_x(uint32_t addr, XF& x) { x.a = lds128(addr), x.b = lds128(addr + 16); }
  static __device__ __forceinline__ void math(const uint4& w, const XF& x, float (&acc)[NCLS][4]) {
    constexpr uint32_t ML = 0x000f000fu, MH = 0x00f000f0u;
    const uint32_t s0 = w.x >> 8, s1 = w.y >> 8, s2 = w.z >> 8, s3 = w.w >> 8;
    mma16816(acc[0], w.x & ML, w.y & ML, s0 & ML, s1 & ML, x.a.x, x.a.y);
    mma16816(acc[1], w.x & MH, w.y & MH, s0 & MH, s1 & MH, x.a.z, x.a.w);
    mma16816(acc[0], w.z & ML, w.w & ML, s2 & ML, s3 & ML, x.b.x, x.b.y);
    mma16816(acc[1], w.z & MH, w.w & MH, s2 & MH, s3 & MH, x.b.z, x.b.w);
  }
  static __device__ __forceinline__ float combine(const float (&a)[NCLS][4], int i) {
    return fmaf(a[1][i], 1.0f / 16.0f, a[0][i]);
  }
};

template <>
struct Codec<2> {
  static constexpr int KBLK = 128, NCLS = 5, LANE_K = 32;
  struct XF { uint4 a, b, c, d; };
  static __device__ __forceinline__ void load_x(uint32_t addr, XF& x) {
    x.a = lds128(addr), x.b = lds128(addr + 16), x.c = lds128(addr + 32), x.d = lds128(addr + 48);
  }
  static __device__ __forceinline__ void math(const uint4& w, const XF& x, float (&acc)[NCLS][4]) {
    constexpr uint32_t M0 = 0x00030003u, M1 = M0 << 2, M2 = M0 << 4, M3 = M0 << 6, M4 = M0 << 8;
    const uint32_t s0 = w.x >> 10, s1 = w.y >> 10, s2 = w.z >> 10, s3 = w.w >> 10;
    mma16816(acc[0], w.x & M0, w.y & M0, s0 & M0, s1 & M0, x.a.x, x.a.y);
    mma16816(acc[1], w.x & M1, w.y & M1, s0 & M1, s1 & M1, x.a.z, x.a.w);
    mma16816(acc[2], w.x & M2, w.y & M2, s0 & M2, s1 & M2, x.b.x, x.b.y);
    mma16816(acc[0], w.z & M0, w.w & M0, s2 & M0, s3 & M0, x.c.x, x.c.y);
    mma16816(acc[1], w.z & M1, w.w & M1, s2 & M1, s3 & M1, x.c.z, x.c.w);
    mma16816(acc[2], w.z & M2, w.w & M2, s2 & M2, s3 & M2, x.d.x, x.d.y);
    mma16816(acc[3], w.x & M3, w.y & M3, w.z & M3, w.w & M3, x.b.z, x.d.z);
    mma16816(acc[4], w.x & M4, w.y & M4, w.z & M4, w.w & M4, x.b.w, x.d.w);
  }
  static __device__ __forceinline__ float combine(const float (&a)[NCLS][4], int i) {
    float v = a[4][i] * (1.0f / 256.0f);
    v = fmaf(a[3][i], 1.0f / 64.0f, v);
    v = fmaf(a[2][i], 1.0f / 16.0f, v);
    v = fmaf(a[1][i], 1.0f / 4.0f, v);
    return v + a[0][i];
  }
};

template <>
struct Codec<3> {
  static constexpr int KBLK = 80, NCLS = 3, LANE_K = 20;
  struct XF { uint2 d0, d1, d2, d3, d4; };
  static __device__ __forceinline__ void load_x(uint32_t addr, XF& x) {
    x.d0 = lds64(addr), x.d1 = lds64(addr + 8), x.d2 = lds64(addr + 16), x.d3 = lds64(addr + 24), x.d4 = lds64(addr + 32);
  }
  static __device__ __forceinline__ void math(const uint4& w, const XF& x, float (&acc)[NCLS][4]) {
    constexpr uint32_t M0 = 0x00070007u, M1 = 0x00380038u, M2 = 0x01c001c0u;
    const uint32_t s0 = w.x >> 9, s1 = w.y >> 9, s2 = w.z >> 9, s3 = w.w >> 9;
    mma16816(acc[0], w.x & M0, w.y & M0, s0 & M0, s1 & M0, x.d0.x, x.d0.y);
    mma16816(acc[1], w.x & M1, w.y & M1, s0 & M1, s1 & M1, x.d1.x, x.d1.y);
    mma16816(acc[0], w.z & M0, w.w & M0, s2 & M0, s3 & M0, x.d2.y, x.d3.x);
    mma16816(acc[1], w.z & M1, w.w & M1, s2 & M1, s3 & M1, x.d3.y, x.d4.x);
    mma16816(acc[2], w.x & M2, w.y & M2, w.z & M2, w.w & M2, x.d2.x, x.d4.y);
  }
  static __device__ __forceinline__ float combine(const float (&a)[NCLS][4], int i) {
    float v = a[2][i] * (1.0f / 64.0f);
    v = fmaf(a[1][i], 1.0f / 8.0f, v);
    return v + a[0][i];
  }
};

template <>
struct Codec<16> {
  static constexpr int KBLK = 16, NCLS = 1, LANE_K = 4;
  struct XF { uint2 a; };
  static __device__ __forceinline__ void load_x(uint32_t addr, XF& x) { x.a = lds64(addr); }
  static __device__ __forceinline__ void math(const uint4& w, const XF& x, float (&acc)[NCLS][4]) {
    mma16816(acc[0], w.x, w.y, w.z, w.w, x.a.x, x.a.y);
  }
  static __device__ __forceinline__ float combine(const float (&a)[NCLS][4], int i) { return a[0][i]; }
};

// ------------------------------------------------------------------------------------------------
// x staging (consumer threads only): residual add, RMSNorm, fp16 rounding points of the reference.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float hsum8(const uint4& v) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    s += f.x;
    s += f.y;
  }
  return s;
}

// residual add of one uint4 (8 halfs), the reference's fp16 add
// sum of the n rank partials of 8 consecutive elements, in rank order, fp32, rounded once (n == 1: the value itself)
__device__ __forceinline__ uint4 rank_sum8(const __half* base, size_t stride, int n, size_t off) {
  uint4 b = ldg_cg_v4(base + off);
  if (n <= 1) return b;
  float acc[8];
  {
    const __half2* h = reinterpret_cast<const __half2*>(&b);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(h[j]);
      acc[2 * j] = f.x, acc[2 * j + 1] = f.y;
    }
  }
  for (int r = 1; r < n; ++r) {
    const uint4 c = ldg_cg_v4(base + (size_t)r * stride + off);
    const __half2* h = reinterpret_cast<const __half2*>(&c);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(h[j]);
      acc[2 * j] += f.x, acc[2 * j + 1] += f.y;
    }
  }
  __half2* o = reinterpret_cast<__half2*>(&b);
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = __floats2half2_rn(acc[2 * j], acc[2 * j + 1]);
  return b;
}

// the residual delta of 8 elements: plain fp16 vector(s) or the LL buffers of the fused tensor-parallel all-reduce
__device__ __forceinline__ uint4 load_delta8(const GemvParams& p, size_t off) {
  if (p.ll_in) {
    unsigned err = 0;
    // once a poll has timed out (error word set) nothing spins again: a broken exchange costs ~2 s once, not per poll
    const unsigned cap = (p.ll_err && *reinterpret_cast<volatile unsigned*>(p.ll_err)) ? 1u : ll::kSpinCap;
    const uint4 v = ll::ll_rank_sum8(reinterpret_cast<const uint8_t*>(p.delta), p.K, p.n_delta, (int)off,
                                     *p.ll_step * (unsigned)p.ll_period + (unsigned)p.ll_in_id + 1u, &err, cap);
    if (err && p.ll_err) *p.ll_err = 1u;
    return v;
  }
  return rank_sum8(p.delta, (size_t)p.K, p.n_delta, off);
}

__device__ __forceinline__ uint4 load_h(const GemvParams& p, int tok, int u) {
  uint4 a = ldg_cg_v4(p.resid + (size_t)tok * p.K + (size_t)u * 8);
  if (p.delta) {
    const uint4 b = load_delta8(p, (size_t)tok * p.K + (size_t)u * 8);
    __half2* ha = reinterpret_cast<__half2*>(&a);
    const __half2* hb = reinterpret_cast<const __half2*>(&b);
#pragma unroll
    for (int j = 0; j < 4; ++j) ha[j] = __hadd2(ha[j], hb[j]);
  }
  return a;
}

// Batched staging (T >= 3).  The CTA-wide path below pays one L2 round trip and one CTA barrier per token; here the
// loads of four tokens are in flight together, the raw residual rows are parked in the x buffer itself, one barrier
// publishes every token's sum of squares, and the normalisation then runs in place out of shared memory.
// Each thread owns the same elements and every sum is formed in the same order as in the per-token path, so the
// staged x, csum and xsum are bit-identical to it: results do not depend on the batch size.
static __device__ void stage_x_batched(const GemvParams& p, int T, const int* cols, __half* xs, float* csum,
                                       float* xsum, float* scratch, int tid) {
  const int nvec = p.K >> 3;
  const int lane = tid & 31, warp = tid >> 5;
  const int iters = (nvec + kConsumerThreads - 1) / kConsumerThreads;  // <= 2 with the RMSNorm prologue (K <= 8192)
  const bool norm = p.pro == B200_PRO_RMSNORM;
  uint4 gv[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
  if (norm) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int u = tid + i * kConsumerThreads;
      if (u < nvec) gv[i] = p.keep_const ? ldg_keep_v4(p.gamma + (size_t)u * 8, l2_policy_evict_last()) : *reinterpret_cast<const uint4*>(p.gamma + (size_t)u * 8);
    }
    constexpr int TB = 4;
    for (int t0 = 0; t0 < T; t0 += TB) {
      uint4 a[TB][2];
#pragma unroll
      for (int j = 0; j < TB; ++j) {
        const int t = min(t0 + j, T - 1);
        const int tok = cols ? cols[t] / p.src_div : t;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int u = tid + i * kConsumerThreads;
          a[j][i] = u < nvec ? load_h(p, tok, u) : make_uint4(0, 0, 0, 0);
        }
      }
#pragma unroll
      for (int j = 0; j < TB; ++j) {
        const int t = t0 + j;
        if (t < T) {  // uniform across the CTA
          const int tok = cols ? cols[t] / p.src_div : t;
          float ssq = 0.f;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int u = tid + i * kConsumerThreads;
            if (u < nvec) {
              if (p.h_out && blockIdx.x == 0)
                *reinterpret_cast<uint4*>(p.h_out + (size_t)tok * p.K + (size_t)u * 8) = a[j][i];
              *reinterpret_cast<uint4*>(xs + (size_t)t * p.x_stride + (size_t)u * 8) = a[j][i];  // raw h, scaled below
              const __half2* h = reinterpret_cast<const __half2*>(&a[j][i]);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 f = __half22float2(h[q]);
                ssq = fmaf(f.x, f.x, ssq);
                ssq = fmaf(f.y, f.y, ssq);
              }
            }
          }
          ssq = warp_sum(ssq);
          if (lane == 0) scratch[t * kConsumerWarps + warp] = ssq;
        }
      }
    }
    named_bar_sync(1, kConsumerThreads);
  }
  if (norm) {
    for (int t = 0; t < T; ++t) {
      float tot = 0.f;
#pragma unroll
      for (int wi = 0; wi < kConsumerWarps; ++wi) tot += scratch[t * kConsumerWarps + wi];
      const float rstd = 1.0f / sqrtf(tot / (float)p.K + p.eps);
      for (int i = 0; i < iters; ++i) {
        const int u = tid + i * kConsumerThreads;
        const bool valid = u < nvec;
        uint4 xo = make_uint4(0, 0, 0, 0);
        if (valid) {
          uint4* slot = reinterpret_cast<uint4*>(xs + (size_t)t * p.x_stride + (size_t)u * 8);
          const uint4 hvi = *slot;  // this thread's own raw h
          const uint4 gm = i == 0 ? gv[0] : gv[1];
          const __half2* h = reinterpret_cast<const __half2*>(&hvi);
          const __half2* gh = reinterpret_cast<const __half2*>(&gm);
          __half2* o = reinterpret_cast<__half2*>(&xo);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 f = __half22float2(h[q]);
            o[q] = __hmul2(__floats2half2_rn(f.x * rstd, f.y * rstd), gh[q]);  // components.py:52-53 rounding points
          }
          *slot = xo;
        }
        float sm = valid ? hsum8(xo) : 0.f;
        sm += __shfl_xor_sync(0xffffffffu, sm, 1);
        sm += __shfl_xor_sync(0xffffffffu, sm, 2);
        sm += __shfl_xor_sync(0xffffffffu, sm, 4);
        if (valid && (lane & 7) == 0) csum[t * p.n_chunk64 + (u >> 3)] = sm;
      }
      for (int k = p.K + tid; k < p.Kpad; k += kConsumerThreads) xs[(size_t)t * p.x_stride + k] = __float2half(0.f);
    }
  } else {
    // Plain activations: the (token, 512-element slice) pairs are walked in batches of 8 loads in flight -- a
    // load -> store -> next-load loop would pay one L2 round trip per pair (32 slots at K = 14336: 128 of them).
    constexpr int PB = 8;
    const int n_pair = T * iters;  // uniform across the CTA (shuffles below)
    for (int q0 = 0; q0 < n_pair; q0 += PB) {
      uint4 xv[PB];
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const int q = min(q0 + j, n_pair - 1);
        const int t = q / iters, i = q - t * iters;
        const int tok = cols ? cols[t] / p.src_div : t;
        const int u = tid + i * kConsumerThreads;
        xv[j] = u < nvec ? ldg_cg_v4(p.xin + (size_t)tok * p.K + (size_t)u * 8) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const int q = q0 + j;
        if (q >= n_pair) break;
        const int t = q / iters, i = q - t * iters;
        const int u = tid + i * kConsumerThreads;
        const bool valid = u < nvec;
        const uint4 xo = valid ? xv[j] : make_uint4(0, 0, 0, 0);
        if (valid) *reinterpret_cast<uint4*>(xs + (size_t)t * p.x_stride + (size_t)u * 8) = xo;
        float sm = valid ? hsum8(xo) : 0.f;
        sm += __shfl_xor_sync(0xffffffffu, sm, 1);
        sm += __shfl_xor_sync(0xffffffffu, sm, 2);
        sm += __shfl_xor_sync(0xffffffffu, sm, 4);
        if (valid && (lane & 7) == 0) csum[t * p.n_chunk64 + (u >> 3)] = sm;
      }
    }
    for (int t = 0; t < T; ++t)
      for (int k = p.K + tid; k < p.Kpad; k += kConsumerThreads) xs[(size_t)t * p.x_stride + k] = __float2half(0.f);
  }
  named_bar_sync(1, kConsumerThreads);
  for (int t = warp; t < T; t += kConsumerWarps) {
    float sm = 0.f;
    for (int c = lane; c < p.n_chunk64; c += 32) sm += csum[t * p.n_chunk64 + c];
    sm = warp_sum(sm);
    if (lane == 0) xsum[t] = sm;
  }
  __syncwarp();
}

static __device__ void stage_x(const GemvParams& p, int T, const int* cols, __half* xs, float* csum, float* xsum,
                        float* scratch, int tid) {
  if (T >= 3) return stage_x_batched(p, T, cols, xs, csum, xsum, scratch, tid);
  const int nvec = p.K >> 3;  // uint4 per row
  const int lane = tid & 31, warp = tid >> 5;
  for (int t = 0; t < T; ++t) {
    const int tok = cols ? cols[t] / p.src_div : t;
    uint4 hv[4], gv[4];
    float rstd = 1.f;
    if (p.pro == B200_PRO_RMSNORM) {
      float ssq = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {  // gamma is a constant: its load overlaps the activation loads below
        const int u = tid + i * kConsumerThreads;
        if (u < nvec) gv[i] = p.keep_const ? ldg_keep_v4(p.gamma + (size_t)u * 8, l2_policy_evict_last()) : *reinterpret_cast<const uint4*>(p.gamma + (size_t)u * 8);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = tid + i * kConsumerThreads;
        if (u < nvec) {
          uint4 a = ldg_cg_v4(p.resid + (size_t)tok * p.K + (size_t)u * 8);
          if (p.delta) {
            const uint4 b = load_delta8(p, (size_t)tok * p.K + (size_t)u * 8);
            __half2* ha = reinterpret_cast<__half2*>(&a);
            const __half2* hb = reinterpret_cast<const __half2*>(&b);
#pragma unroll
            for (int j = 0; j < 4; ++j) ha[j] = __hadd2(ha[j], hb[j]);
          }
          if (p.h_out && blockIdx.x == 0)
            *reinterpret_cast<uint4*>(p.h_out + (size_t)tok * p.K + (size_t)u * 8) = a;
          hv[i] = a;
          const __half2* h = reinterpret_cast<const __half2*>(&a);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            ssq = fmaf(f.x, f.x, ssq);
            ssq = fmaf(f.y, f.y, ssq);
          }
        }
      }
      ssq = warp_sum(ssq);
      if (lane == 0) scratch[t * kConsumerWarps + warp] = ssq;
      named_bar_sync(1, kConsumerThreads);
      float tot = 0.f;
#pragma unroll
      for (int wi = 0; wi < kConsumerWarps; ++wi) tot += scratch[t * kConsumerWarps + wi];
      rstd = 1.0f / sqrtf(tot / (float)p.K + p.eps);
    }
    const int iters = (nvec + kConsumerThreads - 1) / kConsumerThreads;  // uniform trip count (shuffles below)
    if (p.pro != B200_PRO_RMSNORM) {
      // every slice of the row is requested before the first one is used (K = 11008: three loads, one round trip);
      // hv[] is free in this mode
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = tid + i * kConsumerThreads;
        hv[i] = (i < iters && u < nvec) ? ldg_cg_v4(p.xin + (size_t)tok * p.K + (size_t)u * 8) : make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i >= iters) break;
      const int u = tid + i * kConsumerThreads;
      const bool valid = u < nvec;
      uint4 xo = make_uint4(0, 0, 0, 0);
      if (valid) {
        if (p.pro == B200_PRO_RMSNORM) {
          const uint4 gm = i == 0 ? gv[0] : i == 1 ? gv[1] : i == 2 ? gv[2] : gv[3];
          const uint4 hvi = i == 0 ? hv[0] : i == 1 ? hv[1] : i == 2 ? hv[2] : hv[3];
          const __half2* h = reinterpret_cast<const __half2*>(&hvi);
          const __half2* gh = reinterpret_cast<const __half2*>(&gm);
          __half2* o = reinterpret_cast<__half2*>(&xo);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            // fp16(x_f32 * rstd) THEN * weight in fp16 (components.py:52-53)
            o[j] = __hmul2(__floats2half2_rn(f.x * rstd, f.y * rstd), gh[j]);
          }
        } else {
          xo = hv[i];
        }
        *reinterpret_cast<uint4*>(xs + (size_t)t * p.x_stride + (size_t)u * 8) = xo;
      }
      // 64-wide chunk sums of the fp16-rounded x (what the tensor pipe will see)
      float s = valid ? hsum8(xo) : 0.f;
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      if (valid && (lane & 7) == 0) csum[t * p.n_chunk64 + (u >> 3)] = s;
    }
    // zero the k padding (W3: Kpad > K) so padded fields multiply zeros
    for (int k = p.K + tid; k < p.Kpad; k += kConsumerThreads) xs[(size_t)t * p.x_stride + k] = __float2half(0.f);
  }
  named_bar_sync(1, kConsumerThreads);
  for (int t = warp; t < T; t += kConsumerWarps) {
    float s = 0.f;
    for (int c = lane; c < p.n_chunk64; c += 32) s += csum[t * p.n_chunk64 + c];
    s = warp_sum(s);
    if (lane == 0) xsum[t] = s;
  }
  // no trailing barrier: only the epilogue warps read xsum, and they wait on the x_ready mbarrier that every MMA
  // warp arrives on after this function
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// Epilogue role (2 warps): wait for the 8 MMA-warp partials of a tile, reduce in fixed order, apply the
// scales, round to fp16 and run the fused epilogue.  Shared by the TMA-ring and the direct-load kernels.
// ------------------------------------------------------------------------------------------------
template <int BITS, int NT>
__device__ __forceinline__ void epilogue_role(const GemvParams& p, int T, const int* cols, int nta, bool grouped,
                                              int etid, int lane, const float* red, uint64_t* red_full,
                                              uint64_t* red_empty, uint64_t* x_ready, const float* xsum, int& lt,
                                              uint32_t x_par) {
    pdl_wait();
    // positions of this thread's columns (QKV epilogue): loaded once, ahead of every dependent rope load
    int ps_col[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) ps_col[nt] = 0;
    if (p.epi == B200_EPI_QKV) {
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) ps_col[nt] = p.pos[min(nt * 8 + (etid & 7), T - 1)];
    }
    const int tile_begin = (int)(((long long)p.n_tiles * blockIdx.x) / gridDim.x);
    const int tile_end = (int)(((long long)p.n_tiles * (blockIdx.x + 1)) / gridDim.x);
    // Every global load of the epilogue is hoisted out of the per-tile loop: under full-rate weight streaming a
    // single L2/DRAM round trip costs 1-2 us, and a dependent load per tile would throttle the whole CTA to one
    // tile per round trip (the MMA warps may only run two tiles ahead).  Scales and RoPE factors of all local
    // tiles are staged in shared memory once, up front.
    constexpr int kMaxLocal = 16;
    __shared__ __half2 sz_s[kMaxLocal * 16];
    __shared__ float2 rope_s[kMaxLocal * 16];
    const int n_local = tile_end - tile_begin;
    const bool staged = n_local <= kMaxLocal;
    asm volatile("bar.sync 2, %0;" ::"n"(kEpiWarps * 32) : "memory");  // previous phase done with sz_s / rope_s
    if (staged) {
      if (BITS != 16 && !grouped)
        for (int i = etid; i < n_local * 16; i += kEpiWarps * 32) sz_s[i] = p.sz[(size_t)tile_begin * 16 + i];
      if (NT == 1 && p.epi == B200_EPI_QKV)
        for (int i = etid; i < n_local * 16; i += kEpiWarps * 32) {
          const int row = tile_begin * 16 + i;
          const bool rot = row < p.n_q_rows + p.n_kv_rows;
          const int d = (row < p.n_q_rows ? row : row - p.n_q_rows) & 127;
          // column c of this thread is token min(c, T-1); with NT == 1 and T == 1 every column is token 0, for
          // T > 1 the per-column value is fetched below (staging covers the bs = 1 decode fast path)
          rope_s[i] = rot ? p.rope[(size_t)p.pos[0] * 64 + (d >> 1)] : make_float2(1.f, 0.f);
        }
      asm volatile("bar.sync 2, %0;" ::"n"(kEpiWarps * 32) : "memory");
    }
    const bool rope_staged = staged && NT == 1 && T == 1;
    mbar_wait(x_ready, x_par);  // xsum / csum are staged
    const int lt0 = lt;
    for (int tile = tile_begin; tile < tile_end; ++tile, ++lt) {
      const int buf = lt & 1;
      // thread etid owns rows r0 and r0+8 of the tile and column c = etid&7
      const int c = etid & 7, r0 = etid >> 3;  // r0 in 0..7
      __half2 sza = __floats2half2_rn(0.f, 0.f), szb = sza;
      if (BITS != 16 && !grouped) {
        if (staged) {
          sza = sz_s[(lt - lt0) * 16 + r0], szb = sz_s[(lt - lt0) * 16 + r0 + 8];
        } else {
          sza = p.sz[(size_t)tile * 16 + r0], szb = p.sz[(size_t)tile * 16 + r0 + 8];
        }
      }
      float2 cs_pre[NT][2];
      if (p.epi == B200_EPI_QKV) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int row = tile * 16 + r0 + 8 * hh;
          const bool rot = row < p.n_q_rows + p.n_kv_rows;
          const int d = (row < p.n_q_rows ? row : row - p.n_q_rows) & 127;
#pragma unroll
          for (int nt = 0; nt < NT; ++nt)
            cs_pre[nt][hh] = rope_staged ? rope_s[(lt - lt0) * 16 + r0 + 8 * hh]
                                         : (rot ? p.rope[(size_t)ps_col[nt] * 64 + (d >> 1)] : make_float2(1.f, 0.f));
        }
      }
      mbar_wait(&red_full[buf], (lt >> 1) & 1);
      const float* rbase = red + (size_t)buf * kConsumerWarps * (NT * 128);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (nt >= nta) break;
        const int col = nt * 8 + c;
        const int colc = min(col, T - 1);
        float y[2];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int r = r0 + 8 * hh;
          float sum = 0.f;
#pragma unroll
          for (int wi = 0; wi < kConsumerWarps; ++wi) sum += rbase[wi * (NT * 128) + nt * 128 + r * 8 + c];
          if (BITS != 16 && !grouped) {
            const __half2 szv = hh ? szb : sza;
            sum = (__low2float(szv) * kTwo24) * (sum - (__high2float(szv) * kInvTwo24) * xsum[colc]);
          }
          y[hh] = sum;
        }
        if (p.epi == B200_EPI_SILU) {
          // rows r0 (w1) and r0+8 (w3) of the interleaved tile
          const __half a = __float2half_rn(y[0]), b = __float2half_rn(y[1]);
          if (col < T) {
            const float af = __half2float(a);
            const __half sl = __float2half_rn(af / (1.0f + expf(-af)));  // F.silu in fp32, rounded to fp16
            const int orow = cols ? cols[col] : col;
            reinterpret_cast<__half*>(p.out)[(size_t)orow * (p.N >> 1) + tile * 8 + r0] = __hmul(sl, b);
          }
        } else {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int r = r0 + 8 * hh, row = tile * 16 + r;
            const __half y16 = __float2half_rn(y[hh]);
            if (p.epi == B200_EPI_F16) {
              if (col < T) reinterpret_cast<__half*>(p.out)[(size_t)(cols ? cols[col] : col) * p.N + row] = y16;
            } else if (p.epi == B200_EPI_F32) {
              if (col < T) {
                if (p.n_bcast > 0) {  // vocabulary-sharded head: every rank receives this rank's slice of the logits
                  for (int rr = 0; rr < p.n_bcast; ++rr)
                    reinterpret_cast<float*>(p.bcast[rr])[(size_t)p.bcast_off + row] = __half2float(y16);
                } else {
                  reinterpret_cast<float*>(p.out)[(size_t)col * p.N + row] = __half2float(y16);
                }
              }
            } else {  // B200_EPI_QKV
              const float mine = __half2float(y16);
              const float other = __shfl_xor_sync(0xffffffffu, mine, 8);  // row r^1, same column
              const int tok = colc;
              const int ps = ps_col[nt];
              const int brow = (p.t_base + tok) / p.tokens_per_seq;
              const bool is_v = row >= p.n_q_rows + p.n_kv_rows;
              const int local = row < p.n_q_rows ? row : (is_v ? row - p.n_q_rows - p.n_kv_rows : row - p.n_q_rows);
              const int head = local >> 7, d = local & 127;
              float val = mine;
              if (!is_v) {
                // interleaved-pair complex rotation in fp32 (llama.py:67-77), no FMA contraction
                const float2 cs = cs_pre[nt][hh];
                const float xe = (r & 1) ? other : mine, xo = (r & 1) ? mine : other;
                val = (r & 1) ? __fadd_rn(__fmul_rn(xe, cs.y), __fmul_rn(xo, cs.x))
                              : __fsub_rn(__fmul_rn(xe, cs.x), __fmul_rn(xo, cs.y));
              }
              const __half o16 = __float2half_rn(val);
              if (col < T) {
                if (row < p.n_q_rows) {
                  reinterpret_cast<__half*>(p.out)[(size_t)tok * p.n_q_rows + row] = o16;
                } else if (!is_v) {
                  p.kcache[(((size_t)brow * p.hkv + head) * p.cache_seq + ps) * 128 + ((((d >> 3) ^ ((ps & 1) << 2)) << 3) | (d & 7))] = o16;
                } else {
                  p.vtcache[((size_t)brow * p.hkv + head) * p.cache_seq * 128 + (size_t)(ps >> 5) * 4096 + d * 32 + (ps & 31)] = o16;
                }
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&red_empty[buf]);
    }
    if (etid == 0) tl_max(p.tl, 3);
}

// ------------------------------------------------------------------------------------------------
// MMA role (16 warps): consume one GEMV phase.  stage/par (ring position) and lt (tile counter for the
// partial-sum hand-off) persist across phases of a chained launch.
// ------------------------------------------------------------------------------------------------
// (s, z) of the quantisation groups that MMA warp `warp` closes inside ring slot `s` of `tile` (rows g and g + 8).
__device__ __forceinline__ void load_group_scales(const GemvParams& p, int tile, int s, int warp, int g,
                                                  __half2 (&sz)[kChunk][2]) {
  const int blk0 = s * kSlotBlocks + warp * kChunk;
#pragma unroll
  for (int c = 0; c < kChunk; ++c) {
    const int blk = blk0 + c;
    if (blk < p.KB && ((blk + 1) & p.gb_mask) == 0) {
      const int grp = blk >> p.gb_shift;
      const __half2* src = p.sz + ((size_t)tile * p.G + grp) * 16 + g;
      sz[c][0] = __ldg(src);
      sz[c][1] = __ldg(src + 8);
    }
  }
}

// GM: 0 = per-channel scales only, 1 = grouped scales only (compile-time: the per-channel instances carry none of the
// group bookkeeping), 2 = decided at run time from `grouped_rt` (the chained kernel).
template <int BITS, int NT, int GM = 2>
__device__ __forceinline__ void mma_phase(const GemvParams& p, int T, int nta, bool grouped_rt, uint8_t* ring,
                                          uint64_t* full, uint64_t* empty, float* red, uint64_t* red_full,
                                          uint64_t* red_empty, const __half* xs, const float* csum, int& stage,
                                          uint32_t& par, int& lt, int warp, int lane, long long& c_full,
                                          long long& c_red, bool prof) {
  using C = Codec<BITS>;
  const bool grouped = GM == 2 ? grouped_rt : (GM == 1);
  const int tile_begin = (int)(((long long)p.n_tiles * blockIdx.x) / gridDim.x);
  const int tile_end = (int)(((long long)p.n_tiles * (blockIdx.x + 1)) / gridDim.x);
  const int slots_per_tile = (p.KB + kSlotBlocks - 1) / kSlotBlocks;
  const int g = lane >> 2, t4 = lane & 3;
  uint32_t xr[NT];  // 32-bit smem address of the lane's k-run in the staged x row of n-tile nt
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const int row = min(nt * 8 + g, T - 1);
    xr[nt] = smem_u32(xs + (size_t)row * p.x_stride + t4 * C::LANE_K);
  }
  const uint32_t ring32 = smem_u32(ring) + (uint32_t)(warp * kChunk) * 512u + (uint32_t)lane * 16u;
  __half2 szn[kChunk][2];  // scales of the group(s) this warp closes in the NEXT slot (grouped quantisation only)
#pragma unroll
  for (int c = 0; c < kChunk; ++c) szn[c][0] = szn[c][1] = __floats2half2_rn(0.f, 0.f);
  if (grouped && tile_begin < tile_end) load_group_scales(p, tile_begin, 0, warp, g, szn);

  for (int tile = tile_begin; tile < tile_end; ++tile, ++lt) {
    // AS independent accumulator sets (one per k-block of the slot) break the dependent HMMA chains at bs<=8
    constexpr int AS = (NT == 1) ? kChunk : 1;
    float acc[AS][NT][C::NCLS][4];
    float master[NT][4];
#pragma unroll
    for (int a = 0; a < AS; ++a)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int c = 0; c < C::NCLS; ++c)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[a][nt][c][i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) master[nt][i] = 0.f;

    for (int s = 0; s < slots_per_tile; ++s) {
      // grouped scales: this slot's (s, z) pairs were requested one slot ago; request the next slot's now, so the
      // global round trip overlaps a whole slot of math instead of stalling every group flush
      __half2 szc[kChunk][2];
#pragma unroll
      for (int c = 0; c < kChunk; ++c) szc[c][0] = szn[c][0], szc[c][1] = szn[c][1];
      if (grouped) {
        const bool more = s + 1 < slots_per_tile;
        const int tile2 = more ? tile : tile + 1, s2 = more ? s + 1 : 0;
        if (tile2 < tile_end) load_group_scales(p, tile2, s2, warp, g, szn);
      }
      long long c0 = 0;
      if (prof) c0 = clock64();
      mbar_wait(&full[stage], par);
      if (prof) c_full += clock64() - c0;
      const uint32_t wa = ring32 + (uint32_t)stage * kSlotBytes;
      const int blk0 = s * kSlotBlocks + warp * kChunk;
      if (NT == 1 && !grouped && blk0 + kChunk <= p.KB && p.dbg == 0) {
        // ---- fast path (bs <= 8, per-channel scales, full slot): every load issued before the first HMMA ----
        uint4 w[kChunk];
        typename C::XF xf[kChunk];
#pragma unroll
        for (int c = 0; c < kChunk; ++c) w[c] = lds128(wa + c * 512);
#pragma unroll
        for (int c = 0; c < kChunk; ++c) C::load_x(xr[0] + (uint32_t)((blk0 + c) * C::KBLK) * 2u, xf[c]);
#pragma unroll
        for (int c = 0; c < kChunk; ++c) C::math(w[c], xf[c], acc[c % AS][0]);
      } else {
#pragma unroll
        for (int c = 0; c < kChunk; ++c) {
          const int blk = blk0 + c;
          if (blk < p.KB && p.dbg == 0) {
            const uint4 w = lds128(wa + c * 512);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
              if (nt >= nta) break;
              typename C::XF xf;
              C::load_x(xr[nt] + (uint32_t)(blk * C::KBLK) * 2u, xf);
              C::math(w, xf, acc[c % AS][nt]);
            }
            if (grouped && ((blk + 1) & p.gb_mask) == 0) {
              // group boundary: fold this group's integer dot products into the scaled master sum
              const int grp = blk >> p.gb_shift;
              const __half2 sz0 = szc[c][0], sz1 = szc[c][1];
              const float s0 = __low2float(sz0) * kTwo24, z0 = __high2float(sz0) * kInvTwo24;
              const float s1 = __low2float(sz1) * kTwo24, z1 = __high2float(sz1) * kInvTwo24;
#pragma unroll
              for (int nt = 0; nt < NT; ++nt) {
                float gs[2];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const int col = min(nt * 8 + 2 * t4 + j, T - 1);
                  float v = csum[col * p.n_chunk64 + grp * p.gs_chunks];
                  if (p.gs_chunks == 2) v += csum[col * p.n_chunk64 + grp * 2 + 1];
                  gs[j] = v;
                }
                float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int a = 0; a < AS; ++a) {
#pragma unroll
                  for (int i = 0; i < 4; ++i) v[i] += C::combine(acc[a][nt], i);
#pragma unroll
                  for (int cc = 0; cc < C::NCLS; ++cc)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[a][nt][cc][i] = 0.f;
                }
                master[nt][0] = fmaf(s0, v[0] - z0 * gs[0], master[nt][0]);
                master[nt][1] = fmaf(s0, v[1] - z0 * gs[1], master[nt][1]);
                master[nt][2] = fmaf(s1, v[2] - z1 * gs[0], master[nt][2]);
                master[nt][3] = fmaf(s1, v[3] - z1 * gs[1], master[nt][3]);
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
      if (++stage == p.stages) stage = 0, par ^= 1;
    }

    // ---- hand the partial sums to the epilogue warps ----
    const int buf = lt & 1;
    long long c1 = 0;
    if (prof) c1 = clock64();
    mbar_wait(&red_empty[buf], ((lt >> 1) & 1) ^ 1);
    if (prof) c_red += clock64() - c1;
    float* myred = red + ((size_t)buf * kConsumerWarps + warp) * (NT * 128);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      float v0, v1, v2, v3;
      if (grouped) {
        v0 = master[nt][0], v1 = master[nt][1], v2 = master[nt][2], v3 = master[nt][3];
      } else {
        v0 = v1 = v2 = v3 = 0.f;
#pragma unroll
        for (int a = 0; a < AS; ++a) {
          v0 += C::combine(acc[a][nt], 0), v1 += C::combine(acc[a][nt], 1);
          v2 += C::combine(acc[a][nt], 2), v3 += C::combine(acc[a][nt], 3);
        }
      }
      *reinterpret_cast<float2*>(myred + nt * 128 + g * 8 + 2 * t4) = make_float2(v0, v1);
      *reinterpret_cast<float2*>(myred + nt * 128 + (g + 8) * 8 + 2 * t4) = make_float2(v2, v3);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&red_full[buf]);
  }
}

}  // namespace b200
