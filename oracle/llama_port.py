"""ORACLE TEST INFRASTRUCTURE: CPU restatement ("port") of the reference decode path.

A functional PyTorch-CPU restatement of
    Transformer.forward_inference   accessory/model/LLM/llama.py:394-427, mixtral.py:441-474
    TransformerBlock.forward        llama.py:276-288
    Attention.forward (SDPA path)   llama.py:136-208
    FeedForward.forward             llama.py:252-256
    MoE.forward                     mixtral.py:266-294
    RMSNorm (vanilla)               accessory/model/components.py:41-53
    precompute_freqs_cis / apply_rotary_emb / repeat_kv   llama.py:46-89
with the reference's rounding points kept: every linear output, the normalised x before
`* weight`, the RoPE output, the SDPA output, silu(a)*b and both residual adds are
rounded to the model dtype; logits are `output(h[:, -1]).float()`.

It is pinned against the reference itself: tests/test_oracle.py re-runs the unmodified
reference modules live on the same host and compares bit-for-bit (fp16 and fp32), and
compares with the committed outputs of the reference (oracle/make_golden.py ->
tests/golden/*.npz: fp32 bit-for-bit, fp16 to one ulp -- the reference's fp16 CPU GEMM
depends on the host ISA).  This file travels to the GPU box, /root/reference does not.

Tensor parallelism is modelled algebraically (SURVEY.md 8c): `tp` > 1 shards the master
weights exactly like accessory/util/tensor_parallel.py:34-38 and mixtral.py:237, runs the
per-rank partial computations and sums the RowParallel / MoE partial outputs over ranks
(rank order, accumulated in fp32, rounded once -- NCCL's order is unspecified, see DESIGN.md).
"""
import math

import torch
import torch.nn.functional as F


def precompute_freqs_cis(head_dim, end, theta=10000.0, scaling=None):
    """llama.py:46-56 -> complex64 [end, head_dim/2]."""
    inv = 1.0 / (theta ** (torch.arange(0, head_dim, 2)[: head_dim // 2].float() / head_dim))
    t = torch.arange(end)
    if scaling is not None:
        t = t * scaling
    ang = torch.outer(t, inv).float()
    return torch.polar(torch.ones_like(ang), ang)


def rmsnorm(x, weight, eps):
    """components.py:41-53: fp32 norm, cast to x dtype, THEN times weight."""
    xf = x.float()
    n = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
    return n.type_as(x) * weight


def rope(x, freqs_cis):
    """llama.py:59-77: interleaved pairs (2i, 2i+1) as complex, fp32 multiply, cast back.
    x: [B, S, H, hd]; freqs_cis: [S, hd/2] complex64."""
    xc = torch.view_as_complex(x.float().reshape(*x.shape[:-1], -1, 2))
    fc = freqs_cis.view(1, x.shape[1], 1, xc.shape[-1])
    return torch.view_as_real(xc * fc).flatten(3).type_as(x)


def expand_kv(x, n_rep):
    """llama.py:80-89 (repeat_interleave on the head axis)."""
    if n_rep == 1:
        return x
    b, s, h, d = x.shape
    return x[:, :, :, None, :].expand(b, s, h, n_rep, d).reshape(b, s, h * n_rep, d)


def causal_mask(q_len, kv_len, device=None):
    """llama.py:220-224: right-aligned boolean mask."""
    qi = torch.arange(q_len, device=device) - q_len
    ki = torch.arange(kv_len, device=device) - kv_len
    return qi.view(-1, 1) >= ki.view(1, -1)


class PortModel:
    """kind: 'llama' | 'mixtral'.  sd: master (TP=1) state dict, keys per SURVEY.md 8b."""

    def __init__(self, kind, args: dict, sd: dict, dtype=torch.float16, tp: int = 1):
        self.kind, self.a, self.dtype, self.tp = kind, dict(args), dtype, tp
        a = self.a
        self.D, self.L, self.H = a["dim"], a["n_layers"], a["n_heads"]
        self.Hkv = a.get("n_kv_heads") or self.H
        self.hd = self.D // self.H
        self.eps = a.get("norm_eps", 1e-5)
        self.max_seq_len = a.get("max_seq_len", 2048)
        theta = a.get("rope_theta", 10000.0 if kind == "llama" else 1000000.0)
        self.sd = {k: v.to(dtype) for k, v in sd.items()}
        self.device = next(iter(self.sd.values())).device  # the model runs where its weights are (CPU or GPU)
        self.freqs_cis = precompute_freqs_cis(self.hd, self.max_seq_len * 2, theta, a.get("rope_scaling")).to(self.device)
        assert self.H % tp == 0 and self.Hkv % tp == 0
        self.k_cache = self.v_cache = None
        if kind == "mixtral":
            self.E = a["moe"]["num_experts"]
            self.topk = a["moe"]["num_experts_per_tok"]
            assert self.E % tp == 0

    # -- helpers --------------------------------------------------------------------------
    def _w(self, name):
        return self.sd[name]

    def _rank_sum(self, partials):
        """all_reduce(SUM) of model-dtype tensors, modelled in rank order with one rounding."""
        if len(partials) == 1:
            return partials[0]
        acc = partials[0].float()
        for p in partials[1:]:
            acc = acc + p.float()
        return acc.to(partials[0].dtype)

    def alloc_cache(self, bsz):
        shape = (bsz, self.max_seq_len, self.Hkv, self.hd)
        if self.k_cache is None or self.k_cache[0].shape != shape:
            self.k_cache = [torch.zeros(shape, dtype=self.dtype, device=self.device) for _ in range(self.L)]
            self.v_cache = [torch.zeros(shape, dtype=self.dtype, device=self.device) for _ in range(self.L)]

    # -- blocks ---------------------------------------------------------------------------
    def attention(self, i, x, start_pos, fc, causal):
        p = f"layers.{i}.attention."
        B, S, _ = x.shape
        # column-parallel projections: sharding the output rows does not change any value
        q = F.linear(x, self._w(p + "wq.weight")).view(B, S, self.H, self.hd)
        k = F.linear(x, self._w(p + "wk.weight")).view(B, S, self.Hkv, self.hd)
        v = F.linear(x, self._w(p + "wv.weight")).view(B, S, self.Hkv, self.hd)
        q, k = rope(q, fc), rope(k, fc)
        self.k_cache[i][:B, start_pos:start_pos + S] = k
        self.v_cache[i][:B, start_pos:start_pos + S] = v
        keys = self.k_cache[i][:B, :start_pos + S]
        vals = self.v_cache[i][:B, :start_pos + S]
        n_rep = self.H // self.Hkv
        kk = expand_kv(keys, n_rep).transpose(1, 2)
        vv = expand_kv(vals, n_rep).transpose(1, 2)
        mask = causal_mask(S, keys.shape[1], x.device) if causal else None
        o = F.scaled_dot_product_attention(q.transpose(1, 2), kk, vv, dropout_p=0.0, attn_mask=mask)
        o = o.transpose(1, 2).contiguous().view(B, S, -1)
        wo = self._w(p + "wo.weight")
        if self.tp == 1:
            return F.linear(o, wo)
        parts = [F.linear(oc, wc) for oc, wc in zip(o.chunk(self.tp, -1), wo.chunk(self.tp, 1))]
        return self._rank_sum(parts)

    def ffn(self, i, x):
        p = f"layers.{i}.feed_forward."
        w1, w2, w3 = self._w(p + "w1.weight"), self._w(p + "w2.weight"), self._w(p + "w3.weight")
        act = F.silu(F.linear(x, w1)) * F.linear(x, w3)
        if self.tp == 1:
            return F.linear(act, w2)
        parts = [F.linear(ac, wc) for ac, wc in zip(act.chunk(self.tp, -1), w2.chunk(self.tp, 1))]
        return self._rank_sum(parts)

    def moe(self, i, x):
        """mixtral.py:266-294 (inference): fp16 softmax of the gate logits, top-k, renormalise,
        per-expert SwiGLU on the routed tokens, weighted sum over the k slots, all-reduce."""
        p = f"layers.{i}.feed_forward."
        shp = x.shape
        x = x.view(-1, shp[-1])
        scores = F.linear(x, self._w(p + "gate.weight")).softmax(dim=-1).to(x)
        ew, ei = torch.topk(scores, self.topk, dim=-1)
        flat = ei.view(-1)
        ew = ew / ew.sum(dim=-1, keepdim=True)
        xr = x.repeat_interleave(self.topk, dim=0)
        per = self.E // self.tp
        parts = []
        for r in range(self.tp):
            y = torch.zeros_like(xr)
            for e in range(per * r, per * (r + 1)):
                q = p + f"experts.{e}."
                sel = flat == e
                xe = xr[sel]
                act = F.silu(F.linear(xe, self._w(q + "w1.weight"))) * F.linear(xe, self._w(q + "w3.weight"))
                y[sel] = F.linear(act, self._w(q + "w2.weight"))
            parts.append((y.view(*ew.shape, -1) * ew.unsqueeze(-1)).sum(dim=1))
        return self._rank_sum(parts).view(*shp).to(x)

    def block(self, i, x, start_pos, fc, causal):
        p = f"layers.{i}."
        h = x + self.attention(i, rmsnorm(x, self._w(p + "attention_norm.weight"), self.eps), start_pos, fc, causal)
        n = rmsnorm(h, self._w(p + "ffn_norm.weight"), self.eps)
        return h + (self.ffn(i, n) if self.kind == "llama" else self.moe(i, n))

    @torch.inference_mode()
    def forward_inference(self, tokens, start_pos, return_hidden=False):
        """tokens int64 [B, S] -> fp32 logits [B, vocab] of the LAST position (llama.py:425-427)."""
        B, S = tokens.shape
        if start_pos == 0:
            self.alloc_cache(B)
        h = F.embedding(tokens, self._w("tok_embeddings.weight"))
        fc = self.freqs_cis[start_pos:start_pos + S]
        for i in range(self.L):
            h = self.block(i, h, start_pos, fc, causal=(S != 1))
        hn = rmsnorm(h, self._w("norm.weight"), self.eps)
        logits = F.linear(hn[:, -1, :], self._w("output.weight")).float()
        return (logits, h) if return_hidden else logits


# LLaMA-2 / Mixtral public configs (SURVEY.md 8, shape table). 7B = ModelArgs defaults (llama.py:29-43).
CONFIGS = {
    "llama2-7b": dict(kind="llama", dim=4096, n_layers=32, n_heads=32, n_kv_heads=None, multiple_of=256,
                      ffn_dim_multiplier=None, norm_eps=1e-5, rope_theta=10000.0, vocab_size=32000),
    "llama2-13b": dict(kind="llama", dim=5120, n_layers=40, n_heads=40, n_kv_heads=None, multiple_of=256,
                       ffn_dim_multiplier=None, norm_eps=1e-5, rope_theta=10000.0, vocab_size=32000),
    "llama2-70b": dict(kind="llama", dim=8192, n_layers=80, n_heads=64, n_kv_heads=8, multiple_of=4096,
                       ffn_dim_multiplier=1.3, norm_eps=1e-5, rope_theta=10000.0, vocab_size=32000),
    "mixtral-8x7b": dict(kind="mixtral", dim=4096, hidden_dim=14336, n_layers=32, n_heads=32, n_kv_heads=8,
                         norm_eps=1e-5, rope_theta=1000000.0, vocab_size=32000,
                         moe=dict(num_experts=8, num_experts_per_tok=2)),
}
