// Device roles of the bs = 1 integer-tensor-path GEMV (see gemv1.cu for the design notes), written as PHASES that carry
// their ring position / hand-off counters across calls, so that the same code serves the stand-alone kernel (one phase)
// and the persistent whole-step kernel (mega1.cu: one phase after another on a continuously streaming ring).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "gemv_core.cuh"

namespace b200 {

constexpr int kPlanes = 6;
static_assert(kChunk == 2, "the per-warp x staging maps 16 lanes to the warp's pair of k-blocks");

__device__ __forceinline__ void imma16832(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ __half2 h2bits(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }
__device__ __forceinline__ uint32_t bits_h2(__half2 v) { return *reinterpret_cast<uint32_t*>(&v); }

// 8 consecutive fp16 values -> per plane two words of s8 digits: lo word = elements (0,2,1,3), hi word = (4,6,5,7)
// (the byte order of the low / high nibbles of one packed W4 word, pack.cpp kW4Nib).
// Digit p of x is rint(r / 2^(7p-24)) with r the remainder after the higher planes; "x + 1.5*2^(e+10)" rounds x to a
// multiple of 2^e in fp16 and leaves the digit, in two's complement, in the low byte of the sum's bit pattern.
__device__ __forceinline__ void split8(const uint4& xv, uint32_t (&lo)[kPlanes], uint32_t (&hi)[kPlanes]) {
  __half2 r[4] = {h2bits(xv.x), h2bits(xv.y), h2bits(xv.z), h2bits(xv.w)};
  __half2 t[4];
  {  // plane 5 (2^11): the magic constant would overflow fp16, so scale instead; -2048 * d + r is exact in one FMA
    const __half2 sc = h2bits(0x10001000u), mg = h2bits(0x66006600u), ng = h2bits(0xE800E800u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      t[i] = __hfma2(r[i], sc, mg);
      r[i] = __hfma2(__hsub2(t[i], mg), ng, r[i]);
    }
    lo[5] = __byte_perm(bits_h2(t[0]), bits_h2(t[1]), 0x6240);
    hi[5] = __byte_perm(bits_h2(t[2]), bits_h2(t[3]), 0x6240);
  }
#pragma unroll
  for (int p = 4; p >= 1; --p) {
    const uint32_t mb = (uint32_t)(((7 * p + 1) << 10) | 0x200);  // 1.5 * 2^(7p-24+10): exponent field 7p+1
    const __half2 mg = h2bits(mb | (mb << 16));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      t[i] = __hadd2(r[i], mg);
      r[i] = __hsub2(r[i], __hsub2(t[i], mg));
    }
    lo[p] = __byte_perm(bits_h2(t[0]), bits_h2(t[1]), 0x6240);
    hi[p] = __byte_perm(bits_h2(t[2]), bits_h2(t[3]), 0x6240);
  }
  {
    const __half2 mg = h2bits(0x06000600u);  // 1.5 * 2^-14
#pragma unroll
    for (int i = 0; i < 4; ++i) t[i] = __hadd2(r[i], mg);
    lo[0] = __byte_perm(bits_h2(t[0]), bits_h2(t[1]), 0x6240);
    hi[0] = __byte_perm(bits_h2(t[2]), bits_h2(t[3]), 0x6240);
  }
}

// internal prologue code (not part of the C ABI): x = merged split-KV attention partials (mega1.cu)
constexpr int kProAttnMerge = 2;
// Template value "decided at run time from p.pro / p.epi".  The stand-alone kernel (gemv1.cu) is ONE instance for all four
// launches of a layer: with one instance per (prologue, epilogue) pair every launch started on instructions that the 3.5 GB
// of weights streamed since their last use had pushed out of the L2 -- the activation staging alone took ~2.6 us of
// instruction-fetch stalls (profiles/r02s_*).  A shared instance is re-executed every ~10 us and stays cached.
constexpr int kDyn = -1;

// ring position (MMA warps and producer each keep their own copy) + tile counter of the partial-sum hand-off
struct G1State {
  int stage = 0;
  uint32_t par = 0;
  int lt = 0;
};

struct G1Smem {
  uint8_t* ring;
  uint64_t *full, *empty, *red_full, *red_empty;
  int* red;        // [2][kConsumerWarps][128]
  float* scratch;  // [kConsumerWarps]
  uint8_t* xq;     // [kPlanes][xq_stride]
  uint8_t* szr;    // grouped scales: [stages][kSzSlotBytes] (s, z) pairs of the ring slot's groups, copied with the slot
  float* xblk;     // grouped scales: [KB] fp32 sum of the activations of every 64-wide k-block (zero-point term)
};
constexpr int kSzSlotBytes = 2048;  // a ring slot spans 2048 k: 16 groups of 128 (1 KB) or 32 groups of 64 (2 KB), 16 rows x half2

// ------------------------------------------------------------------------------------------------
// MMA warps
// ------------------------------------------------------------------------------------------------
// digit planes of 8 consecutive activations -> shared memory; returns their fp32 sum (for the zero-point term)
__device__ __forceinline__ float stage_piece(const uint4& xo, uint8_t* xq, int xq_stride, int e0) {
  uint32_t lo[kPlanes], hi[kPlanes];
  split8(xo, lo, hi);
#pragma unroll
  for (int pl = 0; pl < kPlanes; ++pl) *reinterpret_cast<uint2*>(xq + (size_t)pl * xq_stride + e0) = make_uint2(lo[pl], hi[pl]);
  return hsum8(xo);
}

// Timeline stamps (b200_timeline / b200_timeline_cta) are off unless a profiling run asks for them: the work sits out of
// line, so that the straight-line code between the dependency wait and the first MMA stays short.  i >= 8: per-CTA only.
static __device__ __noinline__ void g1_stamp_cold(unsigned long long* tl, unsigned long long* tlc, int cta, int i) {
  if (i < 8) tl_max(tl, i);
  tl_cta(tlc, cta, i);
}
__device__ __forceinline__ void g1_stamp(const GemvParams& p, int cta, int i, bool me = threadIdx.x == 0) {
  if (me && (p.tl || p.tlc)) g1_stamp_cold(p.tl, p.tlc, cta, i);
}

// residual delta of 8 elements: a plain fp16 vector at TP = 1; the sum over tensor-parallel ranks (plain or LL buffers,
// load_delta8) runs out of line.  Scalar arguments: a reference to the caller's parameter block would move it to local memory.
static __device__ __noinline__ uint4 g1_delta8_ranks(const __half* delta, int K, int n_delta, int ll_in, const unsigned* ll_step,
                                                     int ll_period, int ll_in_id, unsigned* ll_err, int off) {
  GemvParams q;
  q.delta = delta, q.K = K, q.n_delta = n_delta, q.ll_in = ll_in, q.ll_step = ll_step, q.ll_period = ll_period;
  q.ll_in_id = ll_in_id, q.ll_err = ll_err;
  return load_delta8(q, (size_t)off);
}
__device__ __forceinline__ uint4 g1_delta8(const GemvParams& p, int off) {
  if (!p.ll_in && p.n_delta <= 1) return ldg_cg_v4(p.delta + off);
  return g1_delta8_ranks(p.delta, p.K, p.n_delta, p.ll_in, p.ll_step, p.ll_period, p.ll_in_id, p.ll_err, off);
}

template <int PRO_T, bool GROUPED = false>
__device__ __forceinline__ float stage_own_slice(const GemvParams& p, const G1Smem& sm, int xq_stride, int warp, int lane,
                                                 int slots_per_tile, int cta, bool wait_dep = false) {
  const int PRO = PRO_T == kDyn ? p.pro : PRO_T;
  // lane -> (slot parity, block of the warp's pair, 8-element piece): one 16-byte load covers 8 elements
  const int half = lane >> 4, sub = lane & 15;
  const int n_it = (slots_per_tile + 1) >> 1;
  float xs = 0.f;
  // every load of the slice is in flight before the first conversion (K = 11008: 3 pieces per lane; a dependent
  // load -> convert -> store loop would pay one loaded L2 round trip per piece).  RMSNorm: xv = the residual sums.
  constexpr int kMaxPieces = 4;  // K <= 16384
  constexpr int kMaxIt = 2;      // RMSNorm: K <= 8192 -> <= 4 slots per tile
  uint4 xv[kMaxPieces], gv[kMaxIt];
#pragma unroll
  for (int it = 0; it < kMaxPieces; ++it) xv[it] = make_uint4(0, 0, 0, 0);
  float rstd = 1.f;
  if (PRO == B200_PRO_RMSNORM) {
    float ssq = 0.f;
    bool ok[kMaxIt];
    int e0s[kMaxIt];
#pragma unroll
    for (int it = 0; it < kMaxIt; ++it) {  // the norm weight is a constant: requested before the dependency resolves
      const int s = 2 * it + half;
      const int blk = s * kSlotBlocks + warp * kChunk + (sub >> 3);
      ok[it] = it < n_it && s < slots_per_tile && blk < p.KB;
      e0s[it] = blk * 64 + (sub & 7) * 8;
      gv[it] = make_uint4(0, 0, 0, 0);
      if (ok[it]) gv[it] = p.keep_const ? ldg_keep_v4(p.gamma + e0s[it], l2_policy_evict_last()) : *reinterpret_cast<const uint4*>(p.gamma + e0s[it]);
    }
    if (wait_dep) pdl_wait();
    g1_stamp(p, cta, 4);
#pragma unroll
    for (int it = 0; it < kMaxIt; ++it)
      if (ok[it]) xv[it] = ldg_cg_v4(p.resid + e0s[it]);  // L2-coherent: in the persistent kernel another CTA wrote it this launch
    if (p.delta) {
      uint4 dv[kMaxIt];
#pragma unroll
      for (int it = 0; it < kMaxIt; ++it) dv[it] = ok[it] ? g1_delta8(p, e0s[it]) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int it = 0; it < kMaxIt; ++it) {
        __half2* ha = reinterpret_cast<__half2*>(&xv[it]);
        const __half2* hb = reinterpret_cast<const __half2*>(&dv[it]);
#pragma unroll
        for (int j = 0; j < 4; ++j) ha[j] = __hadd2(ha[j], hb[j]);  // the reference's fp16 residual add
      }
    }
#pragma unroll
    for (int it = 0; it < kMaxIt; ++it) {
      if (ok[it]) {
        if (p.h_out && cta == 0) *reinterpret_cast<uint4*>(p.h_out + e0s[it]) = xv[it];
        const __half2* h = reinterpret_cast<const __half2*>(&xv[it]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(h[j]);
          ssq = fmaf(f.x, f.x, ssq);
          ssq = fmaf(f.y, f.y, ssq);
        }
      }
    }
    ssq = warp_sum(ssq);
    g1_stamp(p, cta, 8);
    if (lane == 0) sm.scratch[warp] = ssq;
    named_bar_sync(1, kConsumerThreads);
    g1_stamp(p, cta, 9);
    float tot = 0.f;
#pragma unroll
    for (int wi = 0; wi < kConsumerWarps; ++wi) tot += sm.scratch[wi];
    rstd = 1.0f / sqrtf(tot / (float)p.K + p.eps);
  }
  if (PRO != B200_PRO_RMSNORM && wait_dep) pdl_wait();
  if (PRO == B200_PRO_NONE) {
#pragma unroll
    for (int it = 0; it < kMaxPieces; ++it) {
      const int s = 2 * it + half;
      const int blk = s * kSlotBlocks + warp * kChunk + (sub >> 3);
      if (it < n_it && s < slots_per_tile && blk < p.KB) xv[it] = ldg_cg_v4(p.xin + blk * 64 + (sub & 7) * 8);
    }
  }
  if (PRO_T == kProAttnMerge) {
    // x = attention output: merge the split-KV partials (m, l, O[128]) of this lane's head in split order, exactly the
    // arithmetic of attn_decode_kernel's merge (exp2 domain), rounded to fp16 like its output (llama.py:191-206).
    // ws layout: O fp32 [Hq][n_split][128] at p.xin, then (m, l) float2 [Hq][n_split] at p.resid; n_split in p.n_slots.
    const float* ws_o = reinterpret_cast<const float*>(p.xin);
    const float2* ws_ml = reinterpret_cast<const float2*>(p.resid);
    const int ns = p.n_slots;
#pragma unroll
    for (int it = 0; it < kMaxPieces; ++it) {
      const int s = 2 * it + half;
      const int blk = s * kSlotBlocks + warp * kChunk + (sub >> 3);
      if (it < n_it && s < slots_per_tile && blk < p.KB) {
        const int e0 = blk * 64 + (sub & 7) * 8, hq = e0 >> 7, d0 = e0 & 127;
        constexpr int kMaxSplit = 8;
        float2 ml[kMaxSplit];
        float4 oa[kMaxSplit], ob[kMaxSplit];
#pragma unroll
        for (int sp = 0; sp < kMaxSplit; ++sp) {  // every load in flight before the first use: one L2 round trip
          ml[sp] = make_float2(-INFINITY, 0.f);
          oa[sp] = ob[sp] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (sp < ns) {
            const float4* src = reinterpret_cast<const float4*>(ws_o + ((size_t)hq * ns + sp) * 128 + d0);
            ml[sp] = __ldcg(&ws_ml[hq * ns + sp]);
            oa[sp] = __ldcg(src), ob[sp] = __ldcg(src + 1);
          }
        }
        float M = -INFINITY;
#pragma unroll
        for (int sp = 0; sp < kMaxSplit; ++sp) M = fmaxf(M, ml[sp].x);
        float L = 0.f, o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = 0.f;
#pragma unroll
        for (int sp = 0; sp < kMaxSplit; ++sp) {
          const float f = (ml[sp].x == -INFINITY) ? 0.f : exp2f(ml[sp].x - M);
          L += ml[sp].y * f;
          o[0] += oa[sp].x * f, o[1] += oa[sp].y * f, o[2] += oa[sp].z * f, o[3] += oa[sp].w * f;
          o[4] += ob[sp].x * f, o[5] += ob[sp].y * f, o[6] += ob[sp].z * f, o[7] += ob[sp].w * f;
        }
        __half2* xo = reinterpret_cast<__half2*>(&xv[it]);
#pragma unroll
        for (int j = 0; j < 4; ++j) xo[j] = __floats2half2_rn(o[2 * j] / L, o[2 * j + 1] / L);
      }
    }
  }
  // conversion, RMSNorm scaling, digit split and plane stores: ONE copy of the code, rolled over the pieces (the piece is
  // picked from the loaded registers by a select chain, nothing goes through local memory); xs sums in piece order
#pragma unroll 1
  for (int it = 0; it < n_it; ++it) {
    const int s = 2 * it + half;
    const int blk = s * kSlotBlocks + warp * kChunk + (sub >> 3);
    const bool valid = s < slots_per_tile && blk < p.KB;
    const int e0 = blk * 64 + (sub & 7) * 8;
    uint4 xo = xv[0];
#pragma unroll
    for (int j = 1; j < kMaxPieces; ++j) xo = it == j ? xv[j] : xo;
    if (valid) {
      if (PRO == B200_PRO_RMSNORM) {
        const uint4 gm = it == 0 ? gv[0] : gv[1];
        const __half2* gh = reinterpret_cast<const __half2*>(&gm);
        __half2* o = reinterpret_cast<__half2*>(&xo);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(o[j]);
          o[j] = __hmul2(__floats2half2_rn(f.x * rstd, f.y * rstd), gh[j]);  // components.py:52-53 rounding points
        }
      }
      xs += hsum8(xo);
      uint32_t lo[kPlanes], hi[kPlanes];
      split8(xo, lo, hi);
#pragma unroll
      for (int pl = 0; pl < kPlanes; ++pl)
        *reinterpret_cast<uint2*>(sm.xq + (size_t)pl * xq_stride + e0) = make_uint2(lo[pl], hi[pl]);
    }
    if (GROUPED) {  // fp32 sum of the 64 activations of this k-block: its 8 pieces sit in 8 adjacent lanes
      float bs = valid ? hsum8(xo) : 0.f;
      bs += __shfl_xor_sync(0xffffffffu, bs, 1);
      bs += __shfl_xor_sync(0xffffffffu, bs, 2);
      bs += __shfl_xor_sync(0xffffffffu, bs, 4);
      if (valid && (sub & 7) == 0) sm.xblk[blk] = bs;
    }
  }
  xs = warp_sum(xs);
  __syncwarp();
  return xs;
}

// The tile loop of a GEMV phase (integer MMAs over the ring slots of this CTA's tiles + hand-off of the exact partial sums);
// xs_w = this warp's partial sum of the activations it staged.
// ARED: the 16 MMA warps ADD their exact integer partial sums into one [16 rows][8 planes] block per hand-off buffer
// (shared-memory atomics; integer addition is order-free, so the result stays deterministic) instead of parking 16
// blocks for the epilogue warps to add up -- at K = 4096 (two ring slots per tile) the two epilogue warps, not the
// MMA warps, set the pace of the main loop (32 LDS + 64 adds per thread and tile).  The warps' sum_k x[k] partials do not
// depend on the tile: they are handed over once (scratch[16 + warp]) and summed in warp order by the epilogue warps.
template <bool GROUPED = false, bool ARED = false>
__device__ __forceinline__ void g1_mma_tiles(const GemvParams& p, const G1Smem& sm, int warp, int lane, int cta, int n_cta,
                                             G1State& st, float xs_w) {
  const int tile_begin = (int)(((long long)p.n_tiles * cta) / n_cta);
  const int tile_end = (int)(((long long)p.n_tiles * (cta + 1)) / n_cta);
  const int slots_per_tile = (p.KB + kSlotBlocks - 1) / kSlotBlocks;
  const int g = lane >> 2, t4 = lane & 3;
  const int xq_stride = (((p.K + 127) >> 7) << 7) + 64;
  const uint32_t xbase = smem_u32(sm.xq) + (uint32_t)min(g, kPlanes - 1) * (uint32_t)xq_stride + (uint32_t)t4 * 16u;
  const uint32_t ring32 = smem_u32(sm.ring) + (uint32_t)(warp * kChunk) * 512u + (uint32_t)lane * 16u;
  constexpr uint32_t ML = 0x0f0f0f0fu, MH = 0xf0f0f0f0u;
  int stage = st.stage, lt = st.lt;
  uint32_t par = st.par;
  // grouped scales: plane weights of this lane's accumulator columns 2*t4, 2*t4+1 (digits in units of 2^(7c-24), the
  // accumulators carry 16 x the sum); columns 6, 7 are spare
  const float pw0 = 2 * t4 < kPlanes ? __int_as_float((127 + 14 * t4 - 28) << 23) : 0.f;
  const float pw1 = 2 * t4 + 1 < kPlanes ? __int_as_float((127 + 14 * t4 + 7 - 28) << 23) : 0.f;
  const int gs = GROUPED ? p.K / p.G : 0;
  for (int tile = tile_begin; tile < tile_end; ++tile, ++lt) {
    float yacc[2] = {0.f, 0.f};  // GROUPED: rows g, g+8 of the tile, this warp's groups (identical in the 4 lanes of a quad)
    int acc[kChunk][2][4];
#pragma unroll
    for (int c = 0; c < kChunk; ++c)
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[c][k][i] = 0;
    for (int s = 0; s < slots_per_tile; ++s) {
      mbar_wait(&sm.full[stage], par);
      if (tile == tile_begin && s == 0) g1_stamp(p, cta, 7);
      const uint32_t wa = ring32 + (uint32_t)stage * kSlotBytes;
      const int blk0 = s * kSlotBlocks + warp * kChunk;
      if (GROUPED) {
#pragma unroll
        for (int c = 0; c < kChunk; ++c)
#pragma unroll
          for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[c][k][i] = 0;
      }
      if (blk0 + kChunk <= p.KB) {
        uint4 w[kChunk], xb[kChunk];
#pragma unroll
        for (int c = 0; c < kChunk; ++c) w[c] = lds128(wa + c * 512);
#pragma unroll
        for (int c = 0; c < kChunk; ++c) xb[c] = lds128(xbase + (uint32_t)(blk0 + c) * 64u);
#pragma unroll
        for (int c = 0; c < kChunk; ++c) {
          imma16832(acc[c][0], w[c].x & ML, w[c].y & ML, w[c].z & ML, w[c].w & ML, xb[c].x, xb[c].z);
          imma16832(acc[c][1], w[c].x & MH, w[c].y & MH, w[c].z & MH, w[c].w & MH, xb[c].y, xb[c].w);
        }
      } else {
#pragma unroll
        for (int c = 0; c < kChunk; ++c) {
          if (blk0 + c < p.KB) {
            const uint4 w = lds128(wa + c * 512);
            const uint4 xb = lds128(xbase + (uint32_t)(blk0 + c) * 64u);
            imma16832(acc[c][0], w.x & ML, w.y & ML, w.z & ML, w.w & ML, xb.x, xb.z);
            imma16832(acc[c][1], w.x & MH, w.y & MH, w.z & MH, w.w & MH, xb.y, xb.w);
          }
        }
      }
      if (GROUPED) {
        // flush this slot's groups: exact integer dots -> fp32 (6 planes), scale and zero point of the group, fp32 running sum
        const uint32_t szb = smem_u32(sm.szr) + (uint32_t)stage * kSzSlotBytes;
        if (gs == 128) {
          if (blk0 < p.KB) {
            int v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = (acc[0][0][i] + acc[1][0][i]) * 16 + (acc[0][1][i] + acc[1][1][i]);
            float f0 = (float)v[0] * pw0 + (float)v[1] * pw1, f1 = (float)v[2] * pw0 + (float)v[3] * pw1;
            f0 += __shfl_xor_sync(0xffffffffu, f0, 1), f1 += __shfl_xor_sync(0xffffffffu, f1, 1);
            f0 += __shfl_xor_sync(0xffffffffu, f0, 2), f1 += __shfl_xor_sync(0xffffffffu, f1, 2);
            const float xg = sm.xblk[blk0] + sm.xblk[blk0 + 1];
            uint32_t a, b;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a) : "r"(szb + (uint32_t)(warp * 16 + g) * 4u));
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(b) : "r"(szb + (uint32_t)(warp * 16 + g + 8) * 4u));
            const __half2 sza = h2bits(a), szb2 = h2bits(b);
            yacc[0] = fmaf(__low2float(sza), f0 - __high2float(sza) * xg, yacc[0]);
            yacc[1] = fmaf(__low2float(szb2), f1 - __high2float(szb2) * xg, yacc[1]);
          }
        } else {  // groups of 64: one k-block each
#pragma unroll
          for (int c = 0; c < kChunk; ++c) {
            if (blk0 + c < p.KB) {
              int v[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) v[i] = acc[c][0][i] * 16 + acc[c][1][i];
              float f0 = (float)v[0] * pw0 + (float)v[1] * pw1, f1 = (float)v[2] * pw0 + (float)v[3] * pw1;
              f0 += __shfl_xor_sync(0xffffffffu, f0, 1), f1 += __shfl_xor_sync(0xffffffffu, f1, 1);
              f0 += __shfl_xor_sync(0xffffffffu, f0, 2), f1 += __shfl_xor_sync(0xffffffffu, f1, 2);
              const float xg = sm.xblk[blk0 + c];
              uint32_t a, b;
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a) : "r"(szb + (uint32_t)((warp * kChunk + c) * 16 + g) * 4u));
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(b) : "r"(szb + (uint32_t)((warp * kChunk + c) * 16 + g + 8) * 4u));
              const __half2 sza = h2bits(a), szb2 = h2bits(b);
              yacc[0] = fmaf(__low2float(sza), f0 - __high2float(sza) * xg, yacc[0]);
              yacc[1] = fmaf(__low2float(szb2), f1 - __high2float(szb2) * xg, yacc[1]);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.empty[stage]);
      if (++stage == p.stages) stage = 0, par ^= 1;
    }
    if (GROUPED) {
      // ---- hand this warp's fp32 partial rows to the epilogue warps (same double-buffered hand-off, floats in place of ints) ----
      const int buf = lt & 1;
      mbar_wait(&sm.red_empty[buf], ((lt >> 1) & 1) ^ 1);
      float* myred = reinterpret_cast<float*>(sm.red) + ((size_t)buf * kConsumerWarps + warp) * 128;
      if (t4 == 0) myred[g] = yacc[0], myred[g + 8] = yacc[1];
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.red_full[buf]);
      continue;
    }
    // ---- hand the exact integer partial sums (x16) to the epilogue warps; column 6 carries sum_k x[k] ----
    int v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int lo = 0, hi = 0;
#pragma unroll
      for (int c = 0; c < kChunk; ++c) lo += acc[c][0][i], hi += acc[c][1][i];
      v[i] = lo * 16 + hi;
    }
    if (ARED) {
      const int buf = lt & 1;
      mbar_wait(&sm.red_empty[buf], ((lt >> 1) & 1) ^ 1);
      int* rb = sm.red + buf * 128;
      if (t4 != 3) {  // columns 6, 7 are spare
        atomicAdd(rb + g * 8 + 2 * t4, v[0]);
        atomicAdd(rb + g * 8 + 2 * t4 + 1, v[1]);
        atomicAdd(rb + (g + 8) * 8 + 2 * t4, v[2]);
        atomicAdd(rb + (g + 8) * 8 + 2 * t4 + 1, v[3]);
      }
      if (lane == 0) sm.scratch[16 + warp] = xs_w;
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.red_full[buf]);
      continue;
    }
    if (t4 == 3) {
      v[0] = v[2] = __float_as_int(xs_w);
      v[1] = v[3] = 0;
    }
    const int buf = lt & 1;
    mbar_wait(&sm.red_empty[buf], ((lt >> 1) & 1) ^ 1);
    int* myred = sm.red + ((size_t)buf * kConsumerWarps + warp) * 128;
    *reinterpret_cast<int2*>(myred + g * 8 + 2 * t4) = make_int2(v[0], v[1]);
    *reinterpret_cast<int2*>(myred + (g + 8) * 8 + 2 * t4) = make_int2(v[2], v[3]);
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.red_full[buf]);
  }
  st.stage = stage, st.par = par, st.lt = lt;
  g1_stamp(p, cta, 2);
  if (threadIdx.x == 0 && p.tlc) p.tlc[(size_t)cta * 16 + 5] = (unsigned long long)(tile_end - tile_begin);
}


// One GEMV phase of the 16 MMA warps of CTA `cta` of `n_cta`.  The caller has made the activations visible
// (griddepcontrol.wait / grid barrier) before the call.
template <int PRO_T, bool GROUPED = false, bool ARED = false>
__device__ __forceinline__ void g1_mma_phase(const GemvParams& p, const G1Smem& sm, int warp, int lane, int cta, int n_cta,
                                             G1State& st, bool wait_dep = false) {
  const int slots_per_tile = (p.KB + kSlotBlocks - 1) / kSlotBlocks;
  const int xq_stride = (((p.K + 127) >> 7) << 7) + 64;  // plane stride = 64 mod 128: planes g, g+1 hit different banks
  const float xs_w = stage_own_slice<PRO_T, GROUPED>(p, sm, xq_stride, warp, lane, slots_per_tile, cta, wait_dep);
  g1_stamp(p, cta, 1);

  g1_mma_tiles<GROUPED, ARED>(p, sm, warp, lane, cta, n_cta, st, xs_w);
}

// Producer side of one GEMV phase: stream this CTA's contiguous tile range through the ring.
__device__ __forceinline__ void g1_producer_phase(const GemvParams& p, const G1Smem& sm, int cta, int n_cta, G1State& st) {
  const int tile_begin = (int)(((long long)p.n_tiles * cta) / n_cta);
  const int tile_end = (int)(((long long)p.n_tiles * (cta + 1)) / n_cta);
  const int slots_per_tile = (p.KB + kSlotBlocks - 1) / kSlotBlocks;
  int stage = st.stage;
  uint32_t par = st.par;
  for (int tile = tile_begin; tile < tile_end; ++tile) {
    const uint8_t* src = p.qw + (size_t)tile * p.KB * 512;
    for (int s = 0; s < slots_per_tile; ++s) {
      mbar_wait(&sm.empty[stage], par ^ 1);
      const int nblk = min(kSlotBlocks, p.KB - s * kSlotBlocks);
      const uint32_t bytes = (uint32_t)nblk * 512u;
      mbar_arrive_expect_tx(&sm.full[stage], bytes);
      bulk_g2s(sm.ring + (size_t)stage * kSlotBytes, src + (size_t)s * kSlotBytes, bytes, &sm.full[stage]);
      if (++stage == p.stages) stage = 0, par ^= 1;
    }
  }
  st.stage = stage, st.par = par;
}

// ------------------------------------------------------------------------------------------------
// Epilogue warps: fixed-order cross-warp reduction (exact in int32), plane recombination in fp32, scales, fused epilogue.
// Thread etid owns rows r0 = etid/8 and r0+8 of a tile and plane column c = etid%8; the 8 lanes of a row group
// exchange their columns with shuffles and then all hold the same y (only c == 0 stores).
// ------------------------------------------------------------------------------------------------
template <int EPI_T, bool GROUPED = false, bool ARED = false>
__device__ __forceinline__ void g1_epilogue_phase(const GemvParams& p, const G1Smem& sm, int etid, int lane, int cta,
                                                  int n_cta, int& lt_io, bool wait_dep = false) {
  const int EPI = EPI_T == kDyn ? p.epi : EPI_T;
  const int tile_begin = (int)(((long long)p.n_tiles * cta) / n_cta);
  const int tile_end = (int)(((long long)p.n_tiles * (cta + 1)) / n_cta);
  constexpr int kMaxLocal = 16;
  __shared__ __half2 sz_s[kMaxLocal * 16];
  __shared__ float2 rope_s[kMaxLocal * 16];
  const int n_local = tile_end - tile_begin;
  const bool staged = n_local <= kMaxLocal;
  asm volatile("bar.sync 2, %0;" ::"n"(kEpiWarps * 32) : "memory");  // the previous phase is done with sz_s / rope_s
  // the scales are constants: their round trip overlaps the wait for the previous kernel (stand-alone launch)
  if (staged && !GROUPED) {
    const uint64_t pol = l2_policy_evict_last();
#pragma unroll 1
    for (int i = etid; i < n_local * 16; i += kEpiWarps * 32)
      sz_s[i] = p.keep_const ? h2bits(ldg_keep_u32(&p.sz[(size_t)tile_begin * 16 + i], pol)) : p.sz[(size_t)tile_begin * 16 + i];
  }
  if (wait_dep) pdl_wait();
  int ps = 0;
  if (EPI == B200_EPI_QKV) ps = p.pos[0];
  if (staged) {
    if (EPI == B200_EPI_QKV)
#pragma unroll 1
      for (int i = etid; i < n_local * 16; i += kEpiWarps * 32) {
        const int row = tile_begin * 16 + i;
        const bool rot = row < p.n_q_rows + p.n_kv_rows;
        const int d = (row < p.n_q_rows ? row : row - p.n_q_rows) & 127;
        rope_s[i] = rot ? p.rope[(size_t)ps * 64 + (d >> 1)] : make_float2(1.f, 0.f);
      }
    asm volatile("bar.sync 2, %0;" ::"n"(kEpiWarps * 32) : "memory");
  }
  g1_stamp(p, cta, 6, etid == 0);
  const int c = etid & 7, r0 = etid >> 3;
  // weight of plane c: digits are in units of 2^(7c-24), the hand-off carries 16 x the sum
  const float pw = c < kPlanes ? __int_as_float((127 + 7 * c - 28) << 23) : 0.f;
  int lt = lt_io;
  float xsum_once = 0.f;
  for (int tile = tile_begin, li = 0; tile < tile_end; ++tile, ++lt, ++li) {
    const int buf = lt & 1;
    __half2 sza = __float2half2_rn(0.f), szb = sza;
    if (!GROUPED) {
      if (staged) {
        sza = sz_s[li * 16 + r0], szb = sz_s[li * 16 + r0 + 8];
      } else {
        sza = p.sz[(size_t)tile * 16 + r0], szb = p.sz[(size_t)tile * 16 + r0 + 8];
      }
    }
    // QKV: the q | k | v boundaries are multiples of the 128-row head, so a 16-row tile lies in one head of one of them;
    // its class, the head offset d0 of row 0 and its destination are decided once per tile
    float2 cs[2];
    int kind = 0, d0 = 0;  // kind: 0 = q, 1 = k, 2 = v
    __half* dst = nullptr;
    if (EPI == B200_EPI_QKV) {
      const int row0 = tile * 16;
      kind = row0 < p.n_q_rows ? 0 : (row0 < p.n_q_rows + p.n_kv_rows ? 1 : 2);
      const int local0 = row0 - (kind == 0 ? 0 : (kind == 1 ? p.n_q_rows : p.n_q_rows + p.n_kv_rows));
      d0 = local0 & 127;
      const size_t hbase = ((size_t)(p.t_base / p.tokens_per_seq) * p.hkv + (local0 >> 7)) * p.cache_seq * 128;
      dst = kind == 0 ? reinterpret_cast<__half*>(p.out) + row0
                      : (kind == 1 ? p.kcache + hbase + (size_t)ps * 128 : p.vtcache + hbase + (size_t)(ps >> 5) * 4096 + (ps & 31));
      const float2* rope_row = p.rope + (size_t)ps * 64;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh)
        cs[hh] = kind == 2 ? make_float2(1.f, 0.f) : (staged ? rope_s[li * 16 + r0 + 8 * hh] : rope_row[(d0 + r0 + 8 * hh) >> 1]);
    }
    mbar_wait(&sm.red_full[buf], (lt >> 1) & 1);
    const int* rbase = sm.red + (size_t)buf * kConsumerWarps * 128;
    float y[2];
    if (ARED && !GROUPED) {
      if (li == 0) {  // the warps' sum_k x[k] partials, same order as the per-tile hand-off sums them
        xsum_once = 0.f;
#pragma unroll
        for (int wi = 0; wi < kConsumerWarps; ++wi) xsum_once += sm.scratch[16 + wi];
      }
      int* rb = sm.red + buf * 128;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int r = r0 + 8 * hh;
        const int isum = rb[r * 8 + c];
        rb[r * 8 + c] = 0;  // ready for the tile after next
        float f = c < kPlanes ? (float)isum * pw : 0.f;
        f += __shfl_xor_sync(0xffffffffu, f, 1);
        f += __shfl_xor_sync(0xffffffffu, f, 2);
        f += __shfl_xor_sync(0xffffffffu, f, 4);
        const __half2 szv = hh ? szb : sza;
        y[hh] = __low2float(szv) * (f - __high2float(szv) * xsum_once);
      }
    } else
    if (GROUPED) {
      // the MMA warps applied the group scales: sum their fp32 rows in a fixed order (warps 2c, 2c+1 here, then the 8 columns)
      const float* rf = reinterpret_cast<const float*>(rbase);
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int r = r0 + 8 * hh;
        float f = rf[(2 * c) * 128 + r] + rf[(2 * c + 1) * 128 + r];
        f += __shfl_xor_sync(0xffffffffu, f, 1);
        f += __shfl_xor_sync(0xffffffffu, f, 2);
        f += __shfl_xor_sync(0xffffffffu, f, 4);
        y[hh] = f;
      }
    } else {
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int r = r0 + 8 * hh;
      int isum = 0;
      float fsum = 0.f;
#pragma unroll
      for (int wi = 0; wi < kConsumerWarps; ++wi) {
        const int vv = rbase[wi * 128 + r * 8 + c];
        isum += vv;
        fsum += __int_as_float(vv);  // meaningful for c == 6 only (the warps' sum_k x[k] partials, fixed order)
      }
      float f = c < kPlanes ? (float)isum * pw : 0.f;
      f += __shfl_xor_sync(0xffffffffu, f, 1);
      f += __shfl_xor_sync(0xffffffffu, f, 2);
      f += __shfl_xor_sync(0xffffffffu, f, 4);
      const float xsum = __shfl_sync(0xffffffffu, fsum, (lane & 24) | 6);
      const __half2 szv = hh ? szb : sza;
      y[hh] = __low2float(szv) * (f - __high2float(szv) * xsum);
    }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.red_empty[buf]);
    if (EPI == B200_EPI_SILU) {
      const __half a = __float2half_rn(y[0]), b = __float2half_rn(y[1]);
      if (c == 0) {
        const float af = __half2float(a);
        const __half sl = __float2half_rn(af / (1.0f + expf(-af)));  // F.silu in fp32, rounded to fp16
        reinterpret_cast<__half*>(p.out)[tile * 8 + r0] = __hmul(sl, b);
      }
    } else {
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int r = r0 + 8 * hh, row = tile * 16 + r;
        const __half y16 = __float2half_rn(y[hh]);
        if (EPI == B200_EPI_F16) {
          if (p.ll_out) {
            // fused all-reduce, push side: rows r0 / r0 ^ 1 sit in lanes 8 apart; the even one stores {half2, seq} to every rank
            const unsigned other = __shfl_xor_sync(0xffffffffu, (unsigned)__half_as_ushort(y16), 8);
            if (c == 0 && (r0 & 1) == 0) {
              const unsigned pay = (unsigned)__half_as_ushort(y16) | (other << 16);
              const unsigned seq = *p.ll_step * (unsigned)p.ll_period + (unsigned)p.ll_out_id + 1u;
#pragma unroll 1
              for (int rr = 0; rr < p.n_bcast; ++rr)
                ll::ll_store(reinterpret_cast<uint8_t*>(p.bcast[rr]) + (size_t)(p.bcast_off + row) * 4, pay, seq);
            }
          } else if (c == 0) {
            if (p.n_bcast > 0) {  // row-parallel partial sums: pushed into every rank's buffer (the all-reduce's data movement)
#pragma unroll 1
              for (int rr = 0; rr < p.n_bcast; ++rr) reinterpret_cast<__half*>(p.bcast[rr])[p.bcast_off + row] = y16;
            } else {
              reinterpret_cast<__half*>(p.out)[row] = y16;
            }
          }
        } else if (EPI == B200_EPI_F32) {
          if (c == 0) reinterpret_cast<float*>(p.out)[row] = __half2float(y16);
        } else {  // B200_EPI_QKV
          const float mine = __half2float(y16);
          const float other = __shfl_xor_sync(0xffffffffu, mine, 8);  // row r^1
          float val = mine;
          if (kind != 2) {
            // interleaved-pair complex rotation in fp32 (llama.py:67-77), no FMA contraction
            const float xe = (r & 1) ? other : mine, xo = (r & 1) ? mine : other;
            val = (r & 1) ? __fadd_rn(__fmul_rn(xe, cs[hh].y), __fmul_rn(xo, cs[hh].x))
                          : __fsub_rn(__fmul_rn(xe, cs[hh].x), __fmul_rn(xo, cs[hh].y));
          }
          const __half o16 = __float2half_rn(val);
          if (c == 0) {
            const int d = d0 + r;
            if (kind == 0) dst[r] = o16;
            else if (kind == 1) dst[(((d >> 3) ^ ((ps & 1) << 2)) << 3) | (d & 7)] = o16;
            else dst[d * 32] = o16;
          }
        }
      }
    }
  }
  lt_io = lt;
  g1_stamp(p, cta, 3, etid == 0);
}

}  // namespace b200
