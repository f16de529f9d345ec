// bs = 1 decode GEMV on the INTEGER tensor path (sm_100a): y = s * (sum_k q[n,k] x[k] - z * sum_k x[k]), exact.
//
// Why a second kernel: at one token per step the fp16 HMMA kernel (gemv.cu) is bound by the ALU work of turning
// packed nibbles into fp16 A fragments (20 SHF/LOP3 per 1024 weights and lane) and by ~4 us of fixed latency per
// launch.  Here
//   * the activation vector is split ONCE per launch into six planes of balanced signed 7-bit digits,
//       x[k] * 2^24 = sum_p d_p[k] * 2^(7p),  d_p in [-64, 64]   (exact for every finite fp16 value),
//     and the six planes ride the N = 8 dimension of IMMA.16832.U8.S8 (columns 6, 7 are spare);
//   * a packed byte holds two nibbles; `w & 0x0f0f0f0f` IS the u8 A register of one IMMA and `w & 0xf0f0f0f0` the
//     A register (16 q) of a second one: 8 LOP3 + 2 IMMA per 1024 weights, no shifts, no conversions;
//   * the dot products are exact int32 sums; planes are recombined in fp32 by the epilogue warps;
//   * every MMA warp stages only the slice of x it consumes itself (no CTA-wide barrier on the activation path;
//     the RMSNorm prologue needs one named barrier for the sum of squares);
//   * the warp's partial sum_k x[k] travels in spare column 6 of the partial-sum hand-off.
// The packed weight format is the one of gemv.cu (csrc/pack.cpp); only the order of x inside a lane's k-run differs.
//
// Reference semantics: F.linear on the OmniQuant fake-quantised weight (SURVEY.md 8c), RMSNorm components.py:41-53,
// RoPE llama.py:59-77, SwiGLU llama.py:252-256.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <string>

#include "gemv1_core.cuh"

namespace b200 {

// ONE instance per scale layout: prologue and epilogue are run-time switches (gemv1_core.cuh, kDyn), so the four GEMV
// launches of a layer execute the same instructions and find them cached.
template <bool GROUPED>
__global__ void __launch_bounds__(kThreads, 1) gemv1_kernel(const __grid_constant__ GemvParams p) {
  const int EPI = p.epi;
  extern __shared__ __align__(128) uint8_t smem[];
  G1Smem sm;
  sm.ring = smem;
  sm.full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * kSlotBytes);
  sm.empty = sm.full + p.stages;
  sm.red_full = sm.empty + p.stages;
  sm.red_empty = sm.red_full + 2;
  sm.red = reinterpret_cast<int*>(sm.red_empty + 2);
  sm.scratch = reinterpret_cast<float*>(sm.red + 2 * kConsumerWarps * 128);
  sm.xq = reinterpret_cast<uint8_t*>(sm.scratch + 32);
  sm.szr = sm.xq + (size_t)kPlanes * ((((p.K + 127) >> 7) << 7) + 64);  // GROUPED only (not allocated otherwise)
  sm.xblk = reinterpret_cast<float*>(sm.szr + (size_t)p.stages * kSzSlotBytes);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], kConsumerWarps);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&sm.red_full[b], kConsumerWarps);
      mbar_init(&sm.red_empty[b], kEpiWarps);
    }
    fence_mbar_init();
  }
  if (tid < 256) sm.red[tid] = 0;  // the two [16][8] blocks the MMA warps add their integer partial sums into
  __syncthreads();
  if (tid == 0) tl_min(p.tl, 0);
  pdl_launch_dependents();
  const int cta = blockIdx.x, n_cta = gridDim.x;
  if (tid == 0) tl_cta(p.tlc, cta, 0);

  if (warp == kConsumerWarps) {
    // ---------------- producer: weight stream, independent of any earlier kernel ----------------
    if (lane == 0) {
      if (cta == 0 && p.const_pf && p.const_pf_bytes > 0) l2_prefetch(p.const_pf, (uint32_t)p.const_pf_bytes & ~15u);
      const int tile_begin = (int)(((long long)p.n_tiles * cta) / n_cta);
      const int tile_end = (int)(((long long)p.n_tiles * (cta + 1)) / n_cta);
      const int slots_per_tile = (p.KB + kSlotBlocks - 1) / kSlotBlocks;
      int stage = 0;
      uint32_t par = 0;
      const uint64_t pol_ef = l2_policy_evict_first();
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const uint8_t* src = p.qw + (size_t)tile * p.KB * 512;
#pragma unroll 1
        for (int s = 0; s < slots_per_tile; ++s) {
          mbar_wait(&sm.empty[stage], par ^ 1);
          const int nblk = min(kSlotBlocks, p.KB - s * kSlotBlocks);
          const uint32_t bytes = (uint32_t)nblk * 512u;
          if (GROUPED) {
            // the (s, z) pairs of the slot's groups travel with the slot: [tile][group][16 rows] half2, contiguous per tile
            const int gs = p.K / p.G;
            const uint32_t sz_bytes = (uint32_t)(nblk * 64 / gs) * 64u;
            const uint8_t* sz_src = reinterpret_cast<const uint8_t*>(p.sz) + ((size_t)tile * p.G + (size_t)s * (kSlotBlocks * 64 / gs)) * 64;
            mbar_arrive_expect_tx(&sm.full[stage], bytes + sz_bytes);
            bulk_g2s(sm.szr + (size_t)stage * kSzSlotBytes, sz_src, sz_bytes, &sm.full[stage]);
          } else {
            mbar_arrive_expect_tx(&sm.full[stage], bytes);
          }
          if (p.stream_ef) bulk_g2s_hint(sm.ring + (size_t)stage * kSlotBytes, src + (size_t)s * kSlotBytes, bytes, &sm.full[stage], pol_ef);
          else bulk_g2s(sm.ring + (size_t)stage * kSlotBytes, src + (size_t)s * kSlotBytes, bytes, &sm.full[stage]);
          if (++stage == p.stages) stage = 0, par ^= 1;
        }
      }
      // own stream fully issued: pull the head of this CTA's region of the NEXT kernel's weights into L2, so HBM keeps
      // streaming through our epilogue, the launch gap and the next kernel's prologue
      if (p.next_w && p.next_bytes > 0)
        prefetch_next_stream(p.next_w, p.next_bytes, p.next_tiles, p.next_grid, p.next_window, cta, n_cta);
      if (EPI == B200_EPI_QKV && p.prefetch_kv) {
        // the attention kernel that follows streams K/V rows [0, pos] of every kv head.  The dependency has long resolved
        // when the last weight slot is issued; the wait makes the pos read exact.
        pdl_wait();
        const int kv_len = min(max(p.pos[0], 0) + 1, p.cache_seq);
        const int brow = p.t_base / p.tokens_per_seq;
        const uint32_t k_bytes = (uint32_t)kv_len * 256u, v_bytes = (uint32_t)((kv_len + 31) >> 5) * 8192u;
        constexpr uint32_t piece = 16384;
        const int kp = (int)((k_bytes + piece - 1) / piece), vp = (int)((v_bytes + piece - 1) / piece);
        const int total = p.hkv * (kp + vp);
#pragma unroll 1
        for (int i = cta; i < total; i += n_cta) {
          const int head = i / (kp + vp), j = i % (kp + vp);
          const size_t base = ((size_t)brow * p.hkv + head) * p.cache_seq * 128;  // halfs, same for K and V
          const bool k = j < kp;
          const uint32_t off = (uint32_t)(k ? j : j - kp) * piece;
          l2_prefetch(reinterpret_cast<const uint8_t*>((k ? p.kcache : p.vtcache) + base) + off, min(piece, (k ? k_bytes : v_bytes) - off));
        }
      }
    }
    return;
  }
  if (warp > kConsumerWarps) {
    int lt = 0;
    g1_epilogue_phase<kDyn, GROUPED, true>(p, sm, tid - (kConsumerWarps + 1) * 32, lane, cta, n_cta, lt, /*wait_dep=*/true);
    return;
  }
  // griddepcontrol.wait happens inside the staging, after the constant loads (norm weight) have been issued
  G1State st;
  g1_mma_phase<kDyn, GROUPED, true>(p, sm, warp, lane, cta, n_cta, st, /*wait_dep=*/true);
}

static size_t g1_smem_bytes(int stages, int xq_stride, bool grouped, int KB) {
  size_t b = (size_t)stages * kSlotBytes + (size_t)stages * 16 + 4 * 8;
  b += (size_t)2 * kConsumerWarps * 128 * 4;
  b += 32 * 4;
  b += (size_t)kPlanes * xq_stride;
  if (grouped) b += (size_t)stages * kSzSlotBytes + (size_t)((KB + 3) & ~3) * 4;  // scale ring + per-k-block activation sums
  return b;
}

template <bool GROUPED>
static int launch1g(const GemvParams& p, int xq_stride, int grid, size_t smem, bool pdl, cudaStream_t st) {
  auto kfn = gemv1_kernel<GROUPED>;
  static size_t configured[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 15;
  if (smem > configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      set_error(std::string("gemv1: cudaFuncSetAttribute: ") + cudaGetErrorString(e));
      return (int)e;
    }
    configured[dev] = smem;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kfn, p);
  if (e != cudaSuccess) {
    set_error(std::string("gemv1: launch: ") + cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

// true when the T = 1 integer-path kernel covers this call (gemv.cu asks before taking its own path)
bool gemv1_supported(const b200_gemv_args_t* a, const GemvParams& p) {
  const int on = tune_get("B200_GEMV1", 1);
  if (!on) return false;
  if (a->T != 1 || p.bits != 4 || p.slot_expert) return false;
  if (p.G != 1) {  // grouped scales: groups of 128 or 64 (a ring slot spans whole groups), flushed per slot by the MMA warps
    const int gs = p.K / p.G;
    if (!tune_get("B200_GEMV1_GROUPED", 1) || (gs != 128 && gs != 64)) return false;
  }
  if (p.pro == B200_PRO_RMSNORM && p.K > 8192) return false;
  return true;
}

int gemv1_launch(const b200_gemv_args_t* a, GemvParams p, cudaStream_t st) {
  const int xq_stride = ((p.K + 127) / 128) * 128 + 64;  // plane stride = 64 mod 128: planes g, g+1 hit different banks
  const size_t cap = std::min<size_t>(smem_optin(), 227 * 1024) - 4096;
  const int ring_kb = tune_get("B200_GEMV_RING_KB", 128);
  // the QKV launch may take a shallower ring so that one attention CTA (96 KB) fits beside it and starts streaming K/V early
  const int qkv_ring_kb = tune_get("B200_QKV_RING_KB", 0);
  const int want_kb = (p.epi == B200_EPI_QKV && qkv_ring_kb > 0) ? qkv_ring_kb : ring_kb;
  int stages = a->ring_bytes > 0 ? a->ring_bytes / kSlotBytes : (want_kb * 1024) / kSlotBytes;
  stages = std::max(2, std::min(stages, 24));
  const bool grouped = p.G > 1;
  while (stages > 2 && g1_smem_bytes(stages, xq_stride, grouped, p.KB) > cap) --stages;
  const size_t smem = g1_smem_bytes(stages, xq_stride, grouped, p.KB);
  if (smem > cap) {
    set_error("gemv1: activation planes do not fit in shared memory (K too large)");
    return B200_E_UNSUPPORTED;
  }
  p.T = 1;
  p.stages = stages;
  p.tl = timeline_slot();
  p.tlc = timeline_cta_slot();
  p.next_w = static_cast<const uint8_t*>(a->prefetch_next);
  p.next_bytes = a->prefetch_bytes;
  p.next_tiles = a->prefetch_tiles;
  p.next_grid = std::min(std::max(a->prefetch_tiles, 1), sm_count());
  p.next_window = prefetch_window_bytes();
  const int pf_kv = tune_get("B200_PF_KV", 1);
  p.prefetch_kv = (p.epi == B200_EPI_QKV && a->prefetch_kv && pf_kv) ? 1 : 0;
  p.keep_const = tune_get("B200_KEEP_CONST", 1);
  p.stream_ef = tune_get("B200_STREAM_EF", 1);
  p.const_pf = tune_get("B200_CONST_PF", 1) ? static_cast<const uint8_t*>(a->prefetch_const) : nullptr;
  p.const_pf_bytes = a->prefetch_const_bytes;
  const int grid = std::min(p.n_tiles, sm_count());
  const bool pdl = a->use_pdl != 0;
  if (p.epi != B200_EPI_F16 && p.epi != B200_EPI_F32 && p.epi != B200_EPI_QKV && p.epi != B200_EPI_SILU) return B200_E_INVAL;
  return p.G > 1 ? launch1g<true>(p, xq_stride, grid, smem, pdl, st) : launch1g<false>(p, xq_stride, grid, smem, pdl, st);
}

}  // namespace b200
