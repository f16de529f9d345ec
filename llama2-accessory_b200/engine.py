"""DecodeEngine: the per-rank driver of the B200 decode hot path.

It owns the packed weights, the KV cache (engine layouts, see kvlayout.py / b200_decode.h: K [B][Hkv][S][128]
chunk-swizzled, V [B][Hkv][S/32][128][32]) and the small activation buffers, and enqueues one decode step as

    embed -> L x [ RMSNorm+QKV+RoPE+KV-append | GQA split-KV attention | wo (+all-reduce)
                   | RMSNorm+gate/up+SiLU*mul | down (+all-reduce) ]          (llama.py:276-288)
          -> RMSNorm + lm_head (fp16) -> fp32 logits                           (llama.py:425-427)

with every residual add folded into the next kernel's prologue, all kernels launched with programmatic
dependent launch and the whole step captured in a CUDA graph.  Mixtral replaces the FFN half by
router -> per-expert gate/up + down -> weighted combine (mixtral.py:266-294).

Tensor parallelism follows the reference (one process per GPU, column-parallel wq/wk/wv/w1/w3/output,
row-parallel wo/w2, whole experts per rank, one all-reduce after each row-parallel linear); the
collectives are NCCL calls on the same stream, captured in the same graph.
"""
import math
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import torch

from . import ops
from .quant import PackedLinear, pack_fp16, pack_quantized, quantize_weight, random_packed

T_MAX = 32


class _DevBytes:
    """A uint8 torch view of device memory the library allocated (b200_ipc_alloc), for the slices the engine reads (logits)."""

    def __init__(self, ptr, nbytes, device):
        self.ptr, self.nbytes = ptr, nbytes
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        self.tensor = torch.as_tensor(self, device=device)


def _os_env(k, d):
    return os.environ.get(k, d)


def llama_ffn_hidden(dim, multiple_of=256, ffn_dim_multiplier=None):
    """llama.py:235-239."""
    h = int(2 * (4 * dim) / 3)
    if ffn_dim_multiplier is not None:
        h = int(ffn_dim_multiplier * h)
    return multiple_of * ((h + multiple_of - 1) // multiple_of)


@dataclass
class EngineConfig:
    kind: str = "llama"            # 'llama' | 'mixtral'
    dim: int = 4096
    n_layers: int = 32
    n_heads: int = 32
    n_kv_heads: Optional[int] = None
    ffn_hidden: int = 11008        # llama: FeedForward hidden; mixtral: expert hidden_dim
    vocab_size: int = 32000
    norm_eps: float = 1e-5
    rope_theta: float = 10000.0
    rope_scaling: Optional[float] = None
    max_seq_len: int = 2048
    max_batch_size: int = 32
    num_experts: int = 0
    experts_per_tok: int = 0
    bits: int = 4                  # 2/3/4, or 16 = unquantised fp16 linears
    group_size: int = 0
    tp_rank: int = 0
    tp_world: int = 1

    @property
    def head_dim(self):
        return self.dim // self.n_heads

    @property
    def kv_heads(self):
        return self.n_kv_heads or self.n_heads

    @classmethod
    def from_model_args(cls, kind, a: dict, **kw):
        if kind == "llama":
            ffn = llama_ffn_hidden(a["dim"], a.get("multiple_of", 256), a.get("ffn_dim_multiplier"))
            theta = a.get("rope_theta", 10000.0)
            ne = nk = 0
        else:
            ffn = a["hidden_dim"]
            theta = a.get("rope_theta", 1000000.0)
            ne, nk = a["moe"]["num_experts"], a["moe"]["num_experts_per_tok"]
        return cls(kind=kind, dim=a["dim"], n_layers=a["n_layers"], n_heads=a["n_heads"],
                   n_kv_heads=a.get("n_kv_heads"), ffn_hidden=ffn, vocab_size=a["vocab_size"],
                   norm_eps=a.get("norm_eps", 1e-5), rope_theta=theta, rope_scaling=a.get("rope_scaling"),
                   max_seq_len=a.get("max_seq_len", 2048), max_batch_size=a.get("max_batch_size", 32),
                   num_experts=ne, experts_per_tok=nk, **kw)


@dataclass
class LayerWeights:
    wqkv: PackedLinear = None
    wo: PackedLinear = None
    attn_norm: torch.Tensor = None
    ffn_norm: torch.Tensor = None
    w13: PackedLinear = None       # llama
    w2: PackedLinear = None
    gate: torch.Tensor = None      # mixtral: fp16 [E, D]
    e_w13: List[PackedLinear] = field(default_factory=list)
    e_w2: List[PackedLinear] = field(default_factory=list)


def rope_table(head_dim, end, theta, scaling):
    """(cos, sin) of precompute_freqs_cis (llama.py:46-56), same torch ops -> same fp32 values."""
    freqs = 1.0 / (theta ** (torch.arange(0, head_dim, 2)[: head_dim // 2].float() / head_dim))
    t = torch.arange(end)
    if scaling is not None:
        t = t * scaling
    ang = torch.outer(t, freqs).float()
    cis = torch.polar(torch.ones_like(ang), ang)
    return torch.stack([cis.real, cis.imag], dim=-1).contiguous().float()  # [end, hd/2, 2]


def _interleave_w13(a, b):
    """rows of w1 and w3 interleaved 8/8 per 16-row tile (EPI_SILU pairs row r with r+8)."""
    n = a.shape[0]
    assert n % 8 == 0 and a.shape == b.shape
    return torch.stack([a.reshape(n // 8, 8, *a.shape[1:]), b.reshape(n // 8, 8, *b.shape[1:])], dim=1).reshape(
        2 * n, *a.shape[1:])


def check_kernel_limits(cfg: "EngineConfig"):
    """Shapes the kernels reject (csrc/gemv.cu build_gemv_params, attn.cu), refused when the engine is built instead of at
    the first launch.  The GEMVs stage one token's activations in shared memory: the RMSNorm prologue takes K = dim <= 8192,
    a plain input K <= 16384 (K = local FFN width for w2, local heads x 128 for wo), so LLaMA2-70B (F = 28672) needs
    TP >= 2; the attention kernel puts the n_rep query heads of a kv head in one MMA tile (<= 16)."""
    tp = max(1, cfg.tp_world)
    if cfg.dim % 128 or cfg.dim > 8192:
        raise ValueError(f"dim = {cfg.dim}: the fused RMSNorm prologue takes multiples of 128 up to 8192")
    f_loc = cfg.ffn_hidden // tp if cfg.kind == "llama" else cfg.ffn_hidden
    if (f_loc + 127) // 128 * 128 > 16384:
        raise ValueError(f"local FFN width {f_loc} > 16384: shard the model over more tensor-parallel ranks "
                         f"(tp_world = {tp}; LLaMA2-70B needs TP >= 2)")
    if cfg.n_heads // tp * cfg.head_dim > 16384:
        raise ValueError("more than 128 local query heads: shard the model over more tensor-parallel ranks")
    n_rep = cfg.n_heads // cfg.kv_heads
    if cfg.n_heads % cfg.kv_heads or n_rep > 16:
        raise ValueError("n_heads must be a multiple of n_kv_heads with at most 16 query heads per kv head")
    if cfg.bits not in (2, 3, 4, 16):
        raise ValueError("bits must be 2, 3, 4 (quantised) or 16 (fp16 linears)")
    if cfg.kind == "mixtral" and not (1 <= cfg.experts_per_tok <= cfg.num_experts):
        raise ValueError("mixtral: need 1 <= experts_per_tok <= num_experts")


class DecodeEngine:
    def __init__(self, cfg: EngineConfig, device="cuda", group=None):
        if cfg.head_dim != 128:
            raise ValueError("the B200 decode kernels are specialised for head_dim = 128")
        if cfg.n_heads % cfg.tp_world or cfg.kv_heads % cfg.tp_world:
            raise ValueError("n_heads and n_kv_heads must be divisible by the tensor-parallel size")
        check_kernel_limits(cfg)
        self.cfg = cfg
        self.device = torch.device(device)
        self.group = group
        self.Hq = cfg.n_heads // cfg.tp_world
        self.Hkv = cfg.kv_heads // cfg.tp_world
        self.F_raw = cfg.ffn_hidden // cfg.tp_world if cfg.kind == "llama" else cfg.ffn_hidden
        # the GEMV streams K in 64..128-wide blocks: pad the local FFN width (e.g. 11008/8 = 1376 -> 1408) with
        # zero weights (rows of w1/w3, columns of w2); the padded activations are exactly 0
        self.F = (self.F_raw + 127) // 128 * 128
        self.V_loc = cfg.vocab_size // cfg.tp_world
        if cfg.kind == "mixtral":
            assert cfg.num_experts % cfg.tp_world == 0
            self.E_loc = cfg.num_experts // cfg.tp_world
            self.e_first = self.E_loc * cfg.tp_rank
        self.t_max = T_MAX if cfg.kind == "llama" else T_MAX // max(1, cfg.experts_per_tok)
        self.layers: List[LayerWeights] = [LayerWeights() for _ in range(cfg.n_layers)]
        self.tok_emb = None
        self.final_norm = None
        self.lm_head: PackedLinear = None
        self.cache_seq = (cfg.max_seq_len + 31) // 32 * 32
        self.rope = rope_table(128, cfg.max_seq_len * 2, cfg.rope_theta, cfg.rope_scaling).to(self.device)
        self.kcache = self.vtcache = None
        self.cache_bsz = 0
        self.use_pdl = True
        self.use_graph = True
        # measurement aid (scripts/shape_bench.py): run ONE rank's shard of a TP > 1 model without the
        # collectives, to time the per-rank kernels of a multi-GPU configuration on a single GPU.  The
        # logits are then partial sums, not the model's -- never set by the product path.
        self.shard_only = False
        # bs = 1, dense LLaMA, TP = 1, per-channel W4: the whole decode step is ONE persistent kernel (csrc/mega1.cu)
        import os as _os
        # B200_MEGA: 0 = separate kernels, 1 = persistent kernel with grid barriers (mega1.cu), 2 = barrier-free dataflow
        # version (mega2.cu)
        _m = int(_os.environ.get("B200_MEGA", "0"))
        self.use_mega = _m != 0
        self.mega_dataflow = _m == 2
        self._mega = None
        self.mega_timeline = None
        # prompts longer than one 32-token chunk: tcgen05 W4A16 GEMM (csrc/prefill.cu) instead of re-streaming the weights
        # once per 32 tokens through the decode GEMV
        self.use_prefill_tc = _os.environ.get("B200_PREFILL_TC", "1") != "0"
        # verification aid: EVERY forward_inference call (single-token steps too) through the tensor-core GEMM, whose dequant
        # stage reproduces the reference's fake-quantised weight fp16(fp16(q - z) * s) bit for bit (tests: strict parity rule)
        self.force_tc = _os.environ.get("B200_FORCE_TC", "0") != "0"
        self._pf = None
        # TP > 1, bs = 1: the all-reduce after wo / w2 is fused into the GEMV kernels (LL push + rank-ordered sum, ll.cuh)
        # instead of 2 NCCL all-reduce kernels per layer
        # verified at TP = 2 on B200 (813 vs 560 tokens/s with NCCL, logits = TP 1 to one fp16 ulp, profiles/r02k_*); bench.py
        # re-checks TP = world against TP = 1 before every timed run and falls back to NCCL if the check fails
        self.use_ar_fused = _os.environ.get("B200_TP_LL", "1") != "0"
        self._ar = None
        # L2 prefetch of the head of every CTA region of the NEXT kernel's weights (+ the K/V rows attention will read) by the
        # producer warps: +2-6 % at bs = 1 once the integer-path GEMV made the step HBM-bound (gpurun_out/r2b_bench.txt)
        self.prefetch_bytes = int(_os_env("B200_PF", "1"))
        self._graphs: Dict[int, tuple] = {}
        self._alloc_buffers()

    # ------------------------------------------------------------------ construction ---------
    def _alloc_buffers(self):
        c, dev, f16 = self.cfg, self.device, torch.float16
        T = T_MAX
        z = lambda *s, dt=f16: torch.zeros(*s, dtype=dt, device=dev)  # noqa: E731
        self.h = [z(T, c.dim), z(T, c.dim)]
        self.q = z(T, self.Hq * 128)
        self.attn = z(T, self.Hq * 128)
        self.o = z(T, c.dim)
        self.f = z(T, c.dim)
        self.act = z(T, self.F)
        self.logits_loc = z(T, self.V_loc, dt=torch.float32)
        self.pos = z(T, dt=torch.int32)
        self.tokens = z(T, dt=torch.int64)
        self.next_tokens = z(T, dt=torch.int64)
        self.counters = z(T * self.Hkv, dt=torch.int32)
        self.ws = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)
        if c.kind == "mixtral":
            ns = T
            self.xn = z(T, c.dim)
            self.slot_w = z(ns)
            self.slot_e = z(ns, dt=torch.int32)
            self.act_slots = z(ns, self.F)
            self.y_slot = z(ns, c.dim)

    def _shard_rows(self, t):
        return t.chunk(self.cfg.tp_world, dim=0)[self.cfg.tp_rank].contiguous()

    def _shard_cols(self, t, unit=1):
        return t.chunk(self.cfg.tp_world, dim=1)[self.cfg.tp_rank].contiguous()

    def _make_linear(self, name, sd, recs, bits, gs, mode, interleave_with=None, cat=None, pad_rows=0, pad_cols=0):
        """Quantise (or take the given record of) the MASTER weight, then shard, then pack.
        mode: 'col' (rows sharded) | 'row' (input features sharded) | 'none'."""
        def one(key):
            if bits == 16:
                w = sd[key].to(torch.float16)
                return ("w", w)
            if recs is not None and key in recs:
                r = recs[key]
                return ("q", r["q"], r["scale"], r["zero"], r["group_size"])
            q, s, z, g = quantize_weight(sd[key], bits, gs)
            return ("q", q, s, z, g)

        def shard(item):
            if item[0] == "w":
                w = item[1]
                return ("w", self._shard_rows(w) if mode == "col" else self._shard_cols(w) if mode == "row" else w)
            _, q, s, z, g = item
            if mode == "col":
                return ("q", self._shard_rows(q), self._shard_rows(s), self._shard_rows(z), g)
            if mode == "row":
                qs = self._shard_cols(q)
                if s.shape[1] > 1 and (s.shape[1] % self.cfg.tp_world or (q.shape[1] // self.cfg.tp_world) % g):
                    raise ValueError(f"row-parallel shard of K={q.shape[1]} over {self.cfg.tp_world} ranks splits a quantisation "
                                     f"group of {g}: pad the layer width or use per-channel scales")
                if s.shape[1] > 1:  # grouped: scales follow the K shard
                    return ("q", qs, self._shard_cols(s), self._shard_cols(z), g)
                return ("q", qs, s, z, qs.shape[1])
            return item

        def pad(item):
            """zero weights: rows (q = 0, s = 0, z = 0) or input columns (q = 0; grouped: extra groups with s = 0)."""
            if not pad_rows and not pad_cols:
                return item
            Fp = torch.nn.functional.pad
            if item[0] == "w":
                return ("w", Fp(item[1], (0, pad_cols, 0, pad_rows)))
            _, q, sc, z, g = item
            q = Fp(q, (0, pad_cols, 0, pad_rows))
            if sc.shape[1] > 1:  # grouped
                assert pad_cols % g == 0
                sc, z = Fp(sc, (0, pad_cols // g, 0, pad_rows)), Fp(z, (0, pad_cols // g, 0, pad_rows))
            else:
                sc, z = Fp(sc, (0, 0, 0, pad_rows)), Fp(z, (0, 0, 0, pad_rows))
                g = q.shape[1]
            return ("q", q, sc, z, g)

        keys = cat if cat is not None else [name]
        items = [pad(shard(one(k))) for k in keys]
        if interleave_with is not None:
            other = pad(shard(one(interleave_with)))
            if items[0][0] == "w":
                items = [("w", _interleave_w13(items[0][1], other[1]))]
            else:
                items = [("q",) + tuple(_interleave_w13(a, b) for a, b in zip(items[0][1:4], other[1:4])) + (items[0][4],)]
        if items[0][0] == "w":
            return pack_fp16(torch.cat([it[1] for it in items], dim=0), self.device)
        q = torch.cat([it[1] for it in items], dim=0)
        s = torch.cat([it[2] for it in items], dim=0)
        z = torch.cat([it[3] for it in items], dim=0)
        g = items[0][4]
        return pack_quantized(q, s, z, bits, 0 if g >= q.shape[1] else g, self.device)

    def load_local_state_dict(self, sd: dict):
        """sd: this rank's shards, exactly what accessory/util/tensor_parallel.py hands to load_state_dict
        (Column [out/TP, in], Row [out, in/TP], Embedding [vocab, D/TP], local experts only).  Quantisation
        is rank-local min/max (DESIGN.md: differs from quantise-master-then-shard only for row-parallel
        per-channel scales)."""
        return self.load_master_state_dict(sd, None, _sharded=True)

    def load_master_state_dict(self, sd: dict, quant_records: Optional[dict] = None, _sharded=False):
        """sd: MASTER (TP=1) fp16 state dict, keys as in SURVEY.md 8b (optionally prefixed 'llma.').
        quant_records: optional {key: dict(q, scale, zero, group_size)} for the quantised linears of the
        master model (e.g. recovered from an OmniQuant checkpoint); otherwise quantised here."""
        c = self.cfg
        col, row = ("none", "none") if _sharded else ("col", "row")
        # plain dicts are re-keyed without the 'llma.' prefix; lazy mappings (checkpoint.LazyMergedStateDict / LazyQuantRecords:
        # one tensor materialised per lookup) already use the bare names and must not be copied
        if isinstance(sd, dict):
            sd = {(k[5:] if k.startswith("llma.") else k): v for k, v in sd.items()}
        if isinstance(quant_records, dict):
            quant_records = {(k[5:] if k.startswith("llma.") else k): v for k, v in quant_records.items()}
        bits, gs, dev = c.bits, c.group_size, self.device
        emb = sd["tok_embeddings.weight"].to(torch.float16).to(dev).contiguous()
        if _sharded and c.tp_world > 1:  # [vocab, D/TP] shards -> full replicated table
            parts = [torch.empty_like(emb) for _ in range(c.tp_world)]
            torch.distributed.all_gather(parts, emb, group=self.group)
            emb = torch.cat(parts, dim=1).contiguous()
        self.tok_emb = emb
        self.final_norm = sd["norm.weight"].to(torch.float16).to(dev).contiguous()
        ow = sd["output.weight"].to(torch.float16)
        self.lm_head = pack_fp16(ow if _sharded else self._shard_rows(ow), dev)
        for i, lw in enumerate(self.layers):
            p = f"layers.{i}."
            lw.attn_norm = sd[p + "attention_norm.weight"].to(torch.float16).to(dev).contiguous()
            lw.ffn_norm = sd[p + "ffn_norm.weight"].to(torch.float16).to(dev).contiguous()
            # fused QKV: every projection is sharded by rows first, then concatenated
            lw.wqkv = self._make_linear(None, sd, quant_records, bits, gs, col,
                                        cat=[p + "attention.wq.weight", p + "attention.wk.weight",
                                             p + "attention.wv.weight"])
            lw.wo = self._make_linear(p + "attention.wo.weight", sd, quant_records, bits, gs, row)
            if c.kind == "llama":
                fpad = self.F - self.F_raw
                lw.w13 = self._make_linear(p + "feed_forward.w1.weight", sd, quant_records, bits, gs, col,
                                           interleave_with=p + "feed_forward.w3.weight", pad_rows=fpad)
                lw.w2 = self._make_linear(p + "feed_forward.w2.weight", sd, quant_records, bits, gs, row, pad_cols=fpad)
            else:
                lw.gate = sd[p + "feed_forward.gate.weight"].to(torch.float16).to(dev).contiguous()
                for e in range(self.e_first, self.e_first + self.E_loc):
                    q = p + f"feed_forward.experts.{e}."
                    lw.e_w13.append(self._make_linear(q + "w1.weight", sd, quant_records, bits, gs, "none",
                                                      interleave_with=q + "w3.weight"))
                    lw.e_w2.append(self._make_linear(q + "w2.weight", sd, quant_records, bits, gs, "none"))
        return self

    def load_random(self, seed=0):
        """Synthetic random-init weights of the configured architecture, generated directly in packed form
        on the device (bench.py: there is no network for checkpoints)."""
        c, dev = self.cfg, self.device
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        D = c.dim
        self.tok_emb = ((torch.rand((c.vocab_size, D), device=dev, generator=g) * 2 - 1) / math.sqrt(D)).half()
        self.final_norm = torch.ones(D, dtype=torch.float16, device=dev)
        self.lm_head = random_packed(16, self.V_loc, D, 0, dev, seed + 1)
        s = seed + 2
        for lw in self.layers:
            lw.attn_norm = torch.ones(D, dtype=torch.float16, device=dev)
            lw.ffn_norm = torch.ones(D, dtype=torch.float16, device=dev)
            lw.wqkv = random_packed(c.bits, (self.Hq + 2 * self.Hkv) * 128, D, c.group_size, dev, s)
            lw.wo = random_packed(c.bits, D, self.Hq * 128, c.group_size, dev, s + 1)
            s += 2
            if c.kind == "llama":
                lw.w13 = random_packed(c.bits, 2 * self.F, D, c.group_size, dev, s)
                lw.w2 = random_packed(c.bits, D, self.F, c.group_size, dev, s + 1)
                s += 2
            else:
                lw.gate = ((torch.rand((c.num_experts, D), device=dev, generator=g) * 2 - 1) * 4 / math.sqrt(D)).half()
                for _ in range(self.E_loc):
                    lw.e_w13.append(random_packed(c.bits, 2 * self.F, D, c.group_size, dev, s))
                    lw.e_w2.append(random_packed(c.bits, D, self.F, c.group_size, dev, s + 1))
                    s += 2
        return self

    # ------------------------------------------------------------------ KV cache -------------
    def allocate_kv_cache(self, bsz: int):
        """llama.py:210-215 semantics: (re)allocate only when the shape changes. Zero-filled: positions
        beyond a sequence's length are multiplied by P = 0 and must be finite."""
        if self.kcache is not None and self.cache_bsz == bsz:
            return
        L, dev = self.cfg.n_layers, self.device
        self.kcache = torch.zeros((L, bsz, self.Hkv, self.cache_seq, 128), dtype=torch.float16, device=dev)
        self.vtcache = torch.zeros((L, bsz, self.Hkv, self.cache_seq // 32, 128, 32), dtype=torch.float16, device=dev)
        self.cache_bsz = bsz
        self._graphs.clear()

    def destroy_kv_cache(self):
        self.kcache = self.vtcache = None
        self.cache_bsz = 0
        self._graphs.clear()

    def fill_kv_cache_noise(self, std=0.5, seed=0):
        """bench.py: pre-fill the cache with N(0, std) noise instead of running a long prefill (SURVEY.md 8d)."""
        g = torch.Generator(device=self.device)
        g.manual_seed(seed)
        self.kcache.normal_(0.0, std, generator=g)
        self.vtcache.normal_(0.0, std, generator=g)

    # ------------------------------------------------------------------ one step -------------
    def _allreduce(self, t, T):
        if self.cfg.tp_world > 1 and not self.shard_only:
            torch.distributed.all_reduce(t[:T], group=self.group)

    def ar_fused_supported(self, T):
        c = self.cfg
        return (self.use_ar_fused and c.tp_world > 1 and not self.shard_only and T == 1 and c.kind == "llama" and c.bits == 4
                and not c.group_size and c.dim <= 8192)

    def _ar_state(self):
        """Peer-mapped LL buffers of the fused all-reduce (CUDA IPC through b200_ipc_*; collective: every rank gets here at its
        first bs = 1 decode step): [2 (wo | w2)][tp_world][dim / 2] 8-byte units per rank, + a local step counter."""
        if self._ar is None:
            import ctypes as C
            c = self.cfg
            one = c.tp_world * c.dim * 4
            pb = self._peer_buffers(2 * one)
            if pb is None:  # no peer mapping on this box: every rank keeps the NCCL all-reduce
                self.use_ar_fused = False
                return None
            own, ptrs = pb
            ctr = torch.zeros(4, dtype=torch.int32, device=self.device)  # [0] decode-step counter, [1] poll time-out flag
            self._ar = dict(own=own, step=ctr, world=c.tp_world, rank=c.tp_rank,
                            peers_o=(C.c_void_p * c.tp_world)(*ptrs),
                            peers_f=(C.c_void_p * c.tp_world)(*[p + one for p in ptrs]),
                            in_o=own, in_f=own + one, period=2 * len(self.layers) + 2)
        return self._ar

    def _ar_args(self, **kw):
        st = self._ar
        d = dict(world=st["world"], rank=st["rank"], step=st["step"].data_ptr(), period=st["period"],
                 err=st["step"].data_ptr() + 4)
        d.update(kw)
        return d

    def check_tp_exchange(self):
        """Fail loudly when a poll of the fused tensor-parallel all-reduce ever timed out (the kernels then continue with
        whatever the buffer held and set this word; ~2 s once, ll.cuh kSpinCap): every logit since is suspect.  One device
        read per prompt (called at start_pos == 0), nothing on the decode path."""
        if self._ar is not None and int(self._ar["step"][1].item()) != 0:
            raise RuntimeError("fused tensor-parallel all-reduce: a rank's partial sums never arrived (peer mapping / NVLink "
                               "problem); restart with B200_TP_LL=0 to use the NCCL all-reduce")

    def _ensure_ws(self, T, n_split):
        need = ops.attn_workspace_bytes(T, self.Hq, n_split)
        if self.ws.numel() < need:
            # captured decode graphs hold the OLD workspace pointer: drop them so that the next decode step re-captures
            # (replaying them after the old block went back to the allocator would corrupt whoever owns it now)
            self.ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
            self._graphs.clear()

    def _layers(self, T, tokens_per_seq, max_kv_len, row0=0):
        """Enqueue all transformer blocks for the T tokens currently in self.h[0] / self.pos."""
        c, pdl = self.cfg, self.use_pdl
        n_split = ops.attn_split(T, self.Hkv, max_kv_len)
        self._ensure_ws(T, n_split)
        cur, delta = 0, None
        PF = self.prefetch_bytes
        fused = self.ar_fused_supported(T)
        if fused:
            st = self._ar_state()
            fused = st is not None
        if fused:
            ops.advance_pos(st["step"], 1, 1)  # one tick per decode step: the sequence numbers of this step's partial sums

        def head(pl):  # (tensor, bytes, tiles) of the next packed weight stream: per-CTA region heads go to L2
            return (pl.qweight, pl.qweight.numel(), pl.N // 16) if (PF and pl is not None) else None
        for i, lw in enumerate(self.layers):
            kc, vt = self.kcache[i, row0:], self.vtcache[i, row0:]
            h_out = self.h[1 - cur] if delta is not None else None
            nxt = self.layers[i + 1].wqkv if i + 1 < len(self.layers) else self.lm_head
            ar_in = self._ar_args(in_buf=st["in_f"], in_id=2 * (i - 1) + 1) if (fused and delta is not None) else None
            ops.gemv(lw.wqkv, T, resid=self.h[cur], delta=delta, h_out=h_out, gamma=lw.attn_norm, eps=c.norm_eps,
                     epilogue=ops.B200_EPI_QKV, out=self.q, use_pdl=pdl, ar=ar_in,
                     qkv=dict(n_q_rows=self.Hq * 128, n_kv_rows=self.Hkv * 128, rope=self.rope, pos=self.pos,
                              tokens_per_seq=tokens_per_seq, kcache=kc, vtcache=vt, cache_seq=self.cache_seq,
                              prefetch_kv=bool(PF)))
            if delta is not None:
                cur = 1 - cur
            ops.attn_decode(self.q, kc, vt, self.pos, self.attn, T=T, Hq=self.Hq, Hkv=self.Hkv,
                            cache_seq=self.cache_seq, tokens_per_seq=tokens_per_seq, max_kv_len=max_kv_len,
                            ws=self.ws, counters=self.counters, n_split=n_split, use_pdl=pdl, prefetch=head(lw.wo))
            if c.kind == "llama":
                nxt_norm = self.layers[i + 1].attn_norm if i + 1 < len(self.layers) else self.final_norm
                ops.gemv(lw.wo, T, xin=self.attn, epilogue=ops.B200_EPI_F16, out=self.o, use_pdl=pdl,
                         prefetch=head(lw.w13), ar=self._ar_args(out_peers=st["peers_o"], out_id=2 * i) if fused else None,
                         prefetch_const=lw.ffn_norm if PF else None)
                if not fused:
                    self._allreduce(self.o, T)
                ops.gemv(lw.w13, T, resid=self.h[cur], delta=self.o, h_out=self.h[1 - cur], gamma=lw.ffn_norm,
                         eps=c.norm_eps, epilogue=ops.B200_EPI_SILU, out=self.act, use_pdl=pdl, prefetch=head(lw.w2),
                         ar=self._ar_args(in_buf=st["in_o"], in_id=2 * i) if fused else None,
                         prefetch_const=nxt_norm if PF else None)
                cur = 1 - cur
                ops.gemv(lw.w2, T, xin=self.act, epilogue=ops.B200_EPI_F16, out=self.f, use_pdl=pdl, prefetch=head(nxt),
                         ar=self._ar_args(out_peers=st["peers_f"], out_id=2 * i + 1) if fused else None)
            else:
                ops.gemv(lw.wo, T, xin=self.attn, epilogue=ops.B200_EPI_F16, out=self.o, use_pdl=pdl)
                self._allreduce(self.o, T)
                k = c.experts_per_tok
                ops.moe_route(T=T, D=c.dim, E=c.num_experts, topk=k, resid=self.h[cur], delta=self.o,
                              h_out=self.h[1 - cur], gamma=lw.ffn_norm, eps=c.norm_eps, gate_w=lw.gate,
                              xn_out=self.xn, slot_weight=self.slot_w, slot_expert=self.slot_e, use_pdl=pdl)
                cur = 1 - cur
                ops.moe_expert_ffn(lw.e_w13, lw.e_w2, T=T, D=c.dim, F=self.F, topk=k, e_first=self.e_first,
                                   xn=self.xn, slot_expert=self.slot_e, act=self.act_slots, y_slot=self.y_slot,
                                   use_pdl=pdl)
                ops.moe_combine(self.y_slot, self.slot_w, self.slot_e, self.f, T=T, D=c.dim, topk=k,
                                e_first=self.e_first, e_count=self.E_loc)
            if not (fused and c.kind == "llama"):
                self._allreduce(self.f, T)
            delta = self.f
        return cur, delta

    def _head(self, T, cur, delta, rows=None):
        """Final RMSNorm + fp16 lm_head -> fp32 logits [n, V] (gathered over TP ranks)."""
        c = self.cfg
        resid, dl, n = self.h[cur], delta, T
        if rows is not None:  # prefill: only the last position of every sequence (llama.py:426)
            resid = resid[:T].index_select(0, rows).contiguous()
            dl = delta[:T].index_select(0, rows).contiguous()
            n = rows.numel()
        ar_in = None
        if rows is None and self.ar_fused_supported(T) and self._ar is not None:
            ar_in = self._ar_args(in_buf=self._ar["in_f"], in_id=2 * (len(self.layers) - 1) + 1)
        ops.gemv(self.lm_head, n, resid=resid, delta=dl, gamma=self.final_norm, eps=c.norm_eps,
                 epilogue=ops.B200_EPI_F32, out=self.logits_loc, use_pdl=self.use_pdl and rows is None, ar=ar_in)
        if c.tp_world == 1 or self.shard_only:
            return self.logits_loc[:n]
        parts = [torch.empty_like(self.logits_loc[:n]) for _ in range(c.tp_world)]
        torch.distributed.all_gather(parts, self.logits_loc[:n].contiguous(), group=self.group)
        return torch.cat(parts, dim=-1)

    def mega_supported(self, T, row0=0, want_logits=True, last_rows=None):
        c = self.cfg
        return (self.use_mega and c.kind == "llama" and T == 1 and c.bits == 4 and not c.group_size
                and want_logits and last_rows is None and row0 == 0 and c.dim <= 8192 and self.F <= 16384
                and self.Hq // self.Hkv <= 8 and c.n_layers <= 96 and self.lm_head is not None and self.lm_head.bits == 16
                and not self.shard_only and c.tp_world <= 8)

    def _peer_buffers(self, nbytes):
        """A zeroed device buffer of nbytes on every rank of the TP group, mapped into every other rank (CUDA IPC, handles
        exchanged with one all_gather over the group).  Returns (own device pointer, [pointer of rank r's buffer for all r]),
        or None on EVERY rank when any rank could not allocate / map (the caller then keeps the NCCL path): every collective
        below is executed by all ranks whatever happened locally, so a failure cannot leave the others waiting."""
        import ctypes as C
        import torch.distributed as dist
        from . import _cabi
        c = self.cfg
        lib = _cabi.lib()
        group = self.group if self.group is not None else dist.group.WORLD
        own = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        ok = lib.b200_ipc_alloc(nbytes, C.byref(own), handle) == 0
        mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device=self.device)
        allh = [torch.empty_like(mine) for _ in range(c.tp_world)]
        dist.all_gather(allh, mine, group=group)
        ptrs = []
        for r in range(c.tp_world):
            if r == c.tp_rank:
                ptrs.append(own.value)
            elif ok:
                hb = (C.c_ubyte * 64)(*allh[r].cpu().tolist())
                peer = C.c_void_p()
                ok = lib.b200_ipc_open(hb, C.byref(peer)) == 0
                ptrs.append(peer.value)
        flag = torch.tensor([1.0 if ok else 0.0], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        torch.cuda.synchronize()
        dist.barrier(group=group)  # every buffer is zeroed and mapped before any rank's kernel can push into it
        if float(flag.item()) < 0.5:
            return None
        return own.value, ptrs

    def _comm_blocks(self, nbytes):
        """The per-rank communication block of the persistent kernel (barrier counters, row-parallel partial sums,
        gathered logits).  tp_world = 1: plain device memory.  tp_world > 1: CUDA-IPC peer-mapped buffers (b200_ipc_*),
        handles exchanged over the tensor-parallel group -- collective, every rank reaches it at its first decode step."""
        c = self.cfg
        if c.tp_world == 1:
            buf = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            return buf, [buf.data_ptr()], None
        pb = self._peer_buffers(nbytes)
        if pb is None:
            raise RuntimeError("persistent kernel at TP > 1: the ranks could not map each other's buffers (CUDA IPC)")
        own, ptrs = pb
        buf = _DevBytes(own, nbytes, self.device)
        return buf.tensor, ptrs, buf

    def _step1_args(self):
        """The C-ABI argument block of b200_decode_step1 for this engine (rebuilt when the KV cache is re-allocated)."""
        from . import _cabi
        import ctypes as C
        key = (self.kcache.data_ptr(), self.vtcache.data_ptr(), self.mega_dataflow)
        if self._mega is not None and self._mega["key"] == key:
            return self._mega["args"]
        c, L = self.cfg, len(self.layers)
        lib = _cabi.lib()
        n_split = lib.b200_step1_choose_split(self.Hkv)
        if self._mega is not None and self._mega["key"][2] == self.mega_dataflow:  # cache re-allocated: keep the block
            comm, comm_ptrs, hdl = self._mega["keep"]["comm"], self._mega["keep"]["comm_ptrs"], self._mega["keep"]["hdl"]
        else:
            nb = (lib.b200_step1_ll_comm_bytes(L, c.dim, self.Hq, self.Hkv, self.F, self.V_loc, c.tp_world) if self.mega_dataflow
                  else lib.b200_step1_comm_bytes(L, c.dim, self.V_loc, c.tp_world))
            comm, comm_ptrs, hdl = self._comm_blocks(nb)
        keep = dict(
            wqkv=(_cabi.Linear * L)(*[lw.wqkv.c_struct() for lw in self.layers]),
            wo=(_cabi.Linear * L)(*[lw.wo.c_struct() for lw in self.layers]),
            w13=(_cabi.Linear * L)(*[lw.w13.c_struct() for lw in self.layers]),
            w2=(_cabi.Linear * L)(*[lw.w2.c_struct() for lw in self.layers]),
            an=(C.c_void_p * L)(*[lw.attn_norm.data_ptr() for lw in self.layers]),
            fn=(C.c_void_p * L)(*[lw.ffn_norm.data_ptr() for lw in self.layers]),
            attn_ws=torch.zeros(lib.b200_step1_attn_ws_bytes(self.Hq, n_split), dtype=torch.uint8, device=self.device),
            comm=comm, comm_ptrs=comm_ptrs, hdl=hdl, comm_arr=(C.c_void_p * c.tp_world)(*comm_ptrs),
        )
        off = (lib.b200_step1_ll_logits_offset(L, c.dim, self.Hq, self.Hkv, self.F, self.V_loc, c.tp_world) if self.mega_dataflow
               else lib.b200_step1_comm_logits_offset(L, c.dim, c.tp_world))
        keep["logits"] = comm[off:off + 4 * self.V_loc * c.tp_world].view(torch.float32).reshape(1, self.V_loc * c.tp_world)
        a = _cabi.Step1Args()
        a.n_layers, a.dim, a.n_heads, a.n_kv_heads, a.ffn = L, c.dim, self.Hq, self.Hkv, self.F
        a.vocab, a.cache_seq, a.eps = self.V_loc, self.cache_seq, c.norm_eps
        a.token, a.tok_emb, a.pos, a.rope = self.tokens.data_ptr(), self.tok_emb.data_ptr(), self.pos.data_ptr(), self.rope.data_ptr()
        a.kcache, a.vtcache = self.kcache.data_ptr(), self.vtcache.data_ptr()
        a.kv_layer_stride = self.kcache.stride(0)
        a.h0, a.h1, a.q, a.act = (t.data_ptr() for t in (self.h[0], self.h[1], self.q, self.act))
        a.attn_ws = keep["attn_ws"].data_ptr()
        a.wqkv, a.wo, a.w13, a.w2 = keep["wqkv"], keep["wo"], keep["w13"], keep["w2"]
        a.attn_norm, a.ffn_norm, a.final_norm = keep["an"], keep["fn"], self.final_norm.data_ptr()
        a.lm_head = self.lm_head.c_struct()
        a.comm, a.tp_world, a.tp_rank = keep["comm_arr"], c.tp_world, c.tp_rank
        a.timeline = self.mega_timeline.data_ptr() if self.mega_timeline is not None else None
        a.n_split, a.use_pdl = n_split, int(self.use_pdl)
        self._mega = dict(key=key, args=a, keep=keep)
        return a

    # ------------------------------------------------------------------ prefill on the tensor cores ----
    T_PREFILL = 256  # tokens per tcgen05 GEMM launch (TMEM: 128 lanes x 256 fp32 columns per CTA)

    def prefill_tc_supported(self):
        """Per-channel W4 dense LLaMA whose linears tile by 128 output rows: prompts go through b200_prefill_gemm_w4."""
        c = self.cfg
        if not self.use_prefill_tc or c.kind != "llama" or c.bits != 4 or c.group_size or self.shard_only:
            return False
        return all(pl.N % 128 == 0 and pl.K % 64 == 0
                   for pl in (self.layers[0].wqkv, self.layers[0].wo, self.layers[0].w13, self.layers[0].w2))

    def _prefill_bufs(self):
        if self._pf is None:
            c, dev, f16 = self.cfg, self.device, torch.float16
            T = self.T_PREFILL
            z = lambda *s: torch.zeros(*s, dtype=f16, device=dev)  # noqa: E731
            self._pf = dict(h=[z(T, c.dim), z(T, c.dim)], x=z(T, c.dim), qkv=z(T, (self.Hq + 2 * self.Hkv) * 128),
                            q=z(T, self.Hq * 128), attn=z(T, self.Hq * 128), o=z(T, c.dim), gu=z(T, 2 * self.F),
                            act=z(T, self.F), f=z(T, c.dim), pos=torch.zeros(T, dtype=torch.int32, device=dev),
                            tok=torch.zeros(T, dtype=torch.int64, device=dev))
        return self._pf

    def _prefill_chunk_tc(self, tokens, pos, tokens_per_seq, row0, max_kv_len, want_rows):
        """One chunk of T <= 256 prompt tokens (nb sequences x tokens_per_seq positions) through every layer: tensor-core
        GEMMs + the elementwise kernels; attention walks the chunk in <= 32-token launches of the decode kernel (each
        token attends to the cache rows [0, pos]).  Returns fp32 logits of `want_rows` (or None)."""
        c, b = self.cfg, self._prefill_bufs()
        T = tokens.numel()
        b["tok"][:T].copy_(tokens)
        b["pos"][:T].copy_(pos)
        ops.embed(b["tok"], self.tok_emb, b["h"][0], T, c.dim, c.vocab_size)
        cur, delta = 0, None
        nq, nkv = self.Hq * 128, self.Hkv * 128
        for i, lw in enumerate(self.layers):
            kc, vt = self.kcache[i, row0:], self.vtcache[i, row0:]
            ops.prefill_rmsnorm(b["h"][cur], delta, b["h"][1 - cur] if delta is not None else None, lw.attn_norm, c.norm_eps,
                                b["x"], T, c.dim)
            if delta is not None:
                cur = 1 - cur
            ops.prefill_gemm_w4(lw.wqkv, b["x"], b["qkv"], T)
            ops.prefill_rope_kv(b["qkv"], b["q"], kc, vt, self.rope, b["pos"], T, nq, nkv, tokens_per_seq, self.cache_seq)
            for t0 in range(0, T, T_MAX):  # sub-chunks stay inside one sequence when tokens_per_seq % 32 == 0 or nb == 1
                tn = min(T_MAX, T - t0)
                tps = tokens_per_seq
                if tokens_per_seq > tn:  # the sub-chunk lies inside one sequence: every token maps to cache row t0 // tokens_per_seq
                    tps = tn
                rb = t0 // tokens_per_seq
                n_split = ops.attn_split(tn, self.Hkv, max_kv_len)
                self._ensure_ws(tn, n_split)
                ops.attn_decode(b["q"][t0:], kc[rb:], vt[rb:], b["pos"][t0:], b["attn"][t0:], T=tn, Hq=self.Hq, Hkv=self.Hkv,
                                cache_seq=self.cache_seq, tokens_per_seq=tps, max_kv_len=max_kv_len, ws=self.ws,
                                counters=self.counters, n_split=n_split, use_pdl=False)
            ops.prefill_gemm_w4(lw.wo, b["attn"], b["o"], T)
            self._allreduce(b["o"], T)
            ops.prefill_rmsnorm(b["h"][cur], b["o"], b["h"][1 - cur], lw.ffn_norm, c.norm_eps, b["x"], T, c.dim)
            cur = 1 - cur
            ops.prefill_gemm_w4(lw.w13, b["x"], b["gu"], T)
            ops.prefill_silu_mul(b["gu"], b["act"], T, self.F)
            ops.prefill_gemm_w4(lw.w2, b["act"], b["f"], T)
            self._allreduce(b["f"], T)
            delta = b["f"]
        if want_rows is None:
            return None
        resid = b["h"][cur][:T].index_select(0, want_rows).contiguous()
        dl = delta[:T].index_select(0, want_rows).contiguous()
        n = want_rows.numel()
        outs = []
        for r0 in range(0, n, T_MAX):  # the fp16 head GEMV takes <= 32 rows per launch
            rn = min(T_MAX, n - r0)
            ops.gemv(self.lm_head, rn, resid=resid[r0:], delta=dl[r0:], gamma=self.final_norm, eps=c.norm_eps,
                     epilogue=ops.B200_EPI_F32, out=self.logits_loc, use_pdl=False)
            lg = self.logits_loc[:rn]
            if c.tp_world > 1 and not self.shard_only:
                parts = [torch.empty_like(lg) for _ in range(c.tp_world)]
                torch.distributed.all_gather(parts, lg.contiguous(), group=self.group)
                lg = torch.cat(parts, dim=-1)
            outs.append(lg.clone())
        return torch.cat(outs, dim=0)

    def _step(self, T, tokens_per_seq, max_kv_len, row0=0, want_logits=True, last_rows=None):
        c = self.cfg
        if self.mega_supported(T, row0, want_logits, last_rows) and self.cache_bsz >= 1:
            a = self._step1_args()
            ops.decode_step1(a, dataflow=self.mega_dataflow)
            return self._mega["keep"]["logits"]  # fp32 [1, vocab] (all ranks' slices: the head's all-gather is in the kernel)
        ops.embed(self.tokens, self.tok_emb, self.h[0], T, self.cfg.dim, self.cfg.vocab_size)
        cur, delta = self._layers(T, tokens_per_seq, max_kv_len, row0)
        if not want_logits:
            return None
        return self._head(T, cur, delta, last_rows)

    # ------------------------------------------------------------------ public API -----------
    @torch.inference_mode()
    def decode_step(self, tokens: torch.Tensor, start_pos: int) -> torch.Tensor:
        """tokens int64 [bsz] (device) at absolute position start_pos -> fp32 logits [bsz, vocab].
        Uses a captured CUDA graph per batch size; `pos` and `tokens` live in static device buffers.
        For bsz <= t_max the result is a VIEW of the graph's static output buffer: the next step overwrites it (clone it to
        keep it; the drop-in Transformer.forward_inference of model/llama_b200.py does, like the reference's fresh tensor,
        llama.py:427)."""
        bsz = tokens.numel()
        if bsz > self.t_max:
            outs = []
            for b0 in range(0, bsz, self.t_max):
                b1 = min(bsz, b0 + self.t_max)
                self.tokens[: b1 - b0].copy_(tokens.reshape(-1)[b0:b1])
                self.pos[: b1 - b0].fill_(start_pos)
                outs.append(self._step(b1 - b0, 1, min(self.cache_seq, (start_pos + 128) // 128 * 128), row0=b0).clone())
            return torch.cat(outs, dim=0)
        self.tokens[:bsz].copy_(tokens.reshape(-1))
        self.pos[:bsz].fill_(start_pos)
        if not self.use_graph:
            return self._step(bsz, 1, min(self.cache_seq, (start_pos + 128) // 128 * 128))
        return self._replay(bsz)

    def _replay(self, bsz):
        if bsz not in self._graphs:
            # warm-up outside capture (cudaFuncSetAttribute, NCCL lazy init), then capture one step
            keep_tok, keep_pos = self.tokens.clone(), self.pos.clone()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._step(bsz, 1, self.cache_seq)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._step(bsz, 1, self.cache_seq)
            self._graphs[bsz] = (g, out)
            self.tokens.copy_(keep_tok)
            self.pos.copy_(keep_pos)
        g, out = self._graphs[bsz]
        g.replay()
        return out

    @torch.inference_mode()
    def capture_greedy_loop(self, bsz: int):
        """One CUDA graph = one full greedy decode step with everything resident on the device:
        step(tokens, pos) -> argmax -> tokens, pos += 1   (meta.py:434-448 without the per-token host sync).
        Returns (graph, launches_per_step). Set self.tokens[:bsz] / self.pos[:bsz] before the first replay.
        After a replay, self.greedy_logits holds that step's fp32 logits [bsz, vocab] (the graph's static output)."""
        def body():
            logits = self._step(bsz, 1, self.cache_seq)
            ops.argmax(logits.contiguous(), self.tokens, bsz, logits.shape[-1])
            ops.advance_pos(self.pos, bsz, 1)
            return logits
        keep_tok, keep_pos = self.tokens.clone(), self.pos.clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            body()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.tokens.copy_(keep_tok)
        self.pos.copy_(keep_pos)
        g = torch.cuda.CUDAGraph()
        n0 = ops.launch_count
        with torch.cuda.graph(g):
            self.greedy_logits = body()
        return g, ops.launch_count - n0

    @torch.inference_mode()
    def forward_inference(self, tokens: torch.Tensor, start_pos: int) -> torch.Tensor:
        """Transformer.forward_inference (llama.py:394-427): tokens int64 [bsz, seqlen] -> fp32 [bsz, vocab]."""
        bsz, seqlen = tokens.shape
        if start_pos + seqlen > self.cfg.max_seq_len:
            raise ValueError(f"sequence position {start_pos + seqlen} exceeds max_seq_len {self.cfg.max_seq_len}")
        if start_pos == 0:
            self.allocate_kv_cache(bsz)
            self.check_tp_exchange()
        if self.kcache is None or bsz > self.cache_bsz:
            raise RuntimeError("KV cache not allocated for this batch size (call with start_pos=0 first)")
        tokens = tokens.to(self.device)
        if seqlen == 1 and not (self.force_tc and self.prefill_tc_supported()):
            return self.decode_step(tokens[:, 0].contiguous(), start_pos)
        # prefill: chunks of <= t_max tokens walk the layer stack in order (each chunk only needs the
        # K/V of earlier chunks); sequences are processed in groups when bsz alone exceeds t_max
        if (seqlen > T_MAX or self.force_tc) and self.prefill_tc_supported():
            # tensor-core prefill: one sequence at a time, chunks of <= 256 positions
            outs = []
            for b0 in range(bsz):
                off, logits = 0, None
                while off < seqlen:
                    ci = min(self.T_PREFILL, seqlen - off)
                    p = torch.arange(start_pos + off, start_pos + off + ci, dtype=torch.int32, device=self.device)
                    last = off + ci >= seqlen
                    rows = torch.tensor([ci - 1], device=self.device) if last else None
                    kv = min(self.cache_seq, (start_pos + off + ci + 127) // 128 * 128)
                    logits = self._prefill_chunk_tc(tokens[b0, off:off + ci], p, ci, b0, kv, rows)
                    off += ci
                outs.append(logits)
            return torch.cat(outs, dim=0)
        outs = []
        gb = min(bsz, self.t_max)
        for b0 in range(0, bsz, gb):
            b1 = min(bsz, b0 + gb)
            nb = b1 - b0
            ci_max = max(1, self.t_max // nb)
            off, logits = 0, None
            while off < seqlen:
                ci = min(ci_max, seqlen - off)
                T = nb * ci
                self.tokens[:T].copy_(tokens[b0:b1, off:off + ci].reshape(-1))
                p = torch.arange(start_pos + off, start_pos + off + ci, dtype=torch.int32, device=self.device)
                self.pos[:T].copy_(p.repeat(nb))
                last = off + ci >= seqlen
                rows = torch.arange(ci - 1, T, ci, device=self.device) if last else None
                kv = min(self.cache_seq, (start_pos + off + ci + 127) // 128 * 128)
                logits = self._step(T, ci, kv, row0=b0, want_logits=last, last_rows=rows)
                off += ci
            outs.append(logits.clone())
        return torch.cat(outs, dim=0)

    @torch.inference_mode()
    def forward_full(self, tokens: torch.Tensor) -> torch.Tensor:
        """Transformer.forward for inference callers (llama.py:373-391, MetaModel.compute_logits):
        causal full-sequence logits [bsz, seqlen, vocab] (model dtype fp16), via chunked prefill."""
        bsz, seqlen = tokens.shape
        if seqlen > self.cfg.max_seq_len:
            raise ValueError("sequence longer than max_seq_len")
        self.allocate_kv_cache(bsz)
        tokens = tokens.to(self.device)
        out = torch.empty((bsz, seqlen, self.cfg.vocab_size), dtype=torch.float16, device=self.device)
        gb = min(bsz, self.t_max)
        for b0 in range(0, bsz, gb):
            b1 = min(bsz, b0 + gb)
            nb = b1 - b0
            ci_max = max(1, self.t_max // nb)
            off = 0
            while off < seqlen:
                ci = min(ci_max, seqlen - off)
                T = nb * ci
                self.tokens[:T].copy_(tokens[b0:b1, off:off + ci].reshape(-1))
                p = torch.arange(off, off + ci, dtype=torch.int32, device=self.device)
                self.pos[:T].copy_(p.repeat(nb))
                kv = min(self.cache_seq, (off + ci + 127) // 128 * 128)
                lg = self._step(T, ci, kv, row0=b0, want_logits=True)
                out[b0:b1, off:off + ci] = lg.reshape(nb, ci, -1).to(torch.float16)
                off += ci
        return out

    # ------------------------------------------------------------------ accounting -----------
    def step_bytes(self, bsz: int, ctx: int) -> dict:
        """Algorithmic HBM bytes of one decode step on this rank (SURVEY.md 8d formula)."""
        c = self.cfg
        w = 0
        for lw in self.layers:
            for pl in (lw.wqkv, lw.wo, lw.w13, lw.w2):
                if pl is not None:
                    w += pl.nbytes
            for pl in lw.e_w13 + lw.e_w2:
                w += pl.nbytes
        head = self.lm_head.nbytes
        kv = 2 * c.n_layers * ctx * self.Hkv * 128 * 2 * bsz
        return {"weights": w, "lm_head": head, "kv": kv, "total": w + head + kv}
