"""ORACLE TEST INFRASTRUCTURE: deterministic synthetic weights and prompts (SURVEY.md 8d).

Every linear / embedding weight ~ U(-1/sqrt(fan_in), +1/sqrt(fan_in)) -- the law of the
reference's `default_linear_init = kaiming_uniform_(a=sqrt(5))` (llama.py:25) -- drawn in
fp32 from a generator seeded by a hash of the tensor NAME (so the value of a tensor does
not depend on module construction order or on which other tensors exist), then cast to
fp16.  RMSNorm weights are 1 + small deterministic perturbation when `perturb_norm` (to
exercise the gamma multiply), else exactly 1 as in components.py:26.
Master (TP=1) tensors are generated once; shards are slices of them.
"""
import hashlib
import math
import zlib

import torch


def llama_ffn_hidden(dim, multiple_of=256, ffn_dim_multiplier=None):
    """llama.py:235-239."""
    h = int(2 * (4 * dim) / 3)
    if ffn_dim_multiplier is not None:
        h = int(ffn_dim_multiplier * h)
    return multiple_of * ((h + multiple_of - 1) // multiple_of)


def _gen(name, seed):
    g = torch.Generator()
    g.manual_seed((zlib.crc32(name.encode()) ^ (seed * 0x9E3779B1)) & 0x7FFFFFFF)
    return g


def _uniform(name, shape, fan_in, seed, gain=1.0):
    b = gain / math.sqrt(fan_in)
    w = torch.rand(shape, generator=_gen(name, seed), dtype=torch.float32)
    return ((w * 2.0 - 1.0) * b).to(torch.float16)


def _norm_weight(name, dim, seed, perturb):
    if not perturb:
        return torch.ones(dim, dtype=torch.float16)
    w = torch.rand(dim, generator=_gen(name, seed), dtype=torch.float32)
    return (1.0 + 0.25 * (w - 0.5)).to(torch.float16)


def llama_state_dict(args: dict, seed: int = 0, perturb_norm: bool = True, gain: float = 1.0):
    """Keys as in SURVEY.md 8b (no `llma.` prefix). args: dict of llama ModelArgs fields."""
    D, L, H = args["dim"], args["n_layers"], args["n_heads"]
    Hkv = args.get("n_kv_heads") or H
    hd = D // H
    V = args["vocab_size"]
    F = llama_ffn_hidden(D, args.get("multiple_of", 256), args.get("ffn_dim_multiplier"))
    sd = {"tok_embeddings.weight": _uniform("tok_embeddings.weight", (V, D), D, seed)}
    for i in range(L):
        p = f"layers.{i}."
        sd[p + "attention.wq.weight"] = _uniform(p + "wq", (H * hd, D), D, seed, gain)
        sd[p + "attention.wk.weight"] = _uniform(p + "wk", (Hkv * hd, D), D, seed, gain)
        sd[p + "attention.wv.weight"] = _uniform(p + "wv", (Hkv * hd, D), D, seed, gain)
        sd[p + "attention.wo.weight"] = _uniform(p + "wo", (D, H * hd), H * hd, seed, gain)
        sd[p + "feed_forward.w1.weight"] = _uniform(p + "w1", (F, D), D, seed, gain)
        sd[p + "feed_forward.w2.weight"] = _uniform(p + "w2", (D, F), F, seed, gain)
        sd[p + "feed_forward.w3.weight"] = _uniform(p + "w3", (F, D), D, seed, gain)
        sd[p + "attention_norm.weight"] = _norm_weight(p + "an", D, seed, perturb_norm)
        sd[p + "ffn_norm.weight"] = _norm_weight(p + "fn", D, seed, perturb_norm)
    sd["norm.weight"] = _norm_weight("norm", D, seed, perturb_norm)
    sd["output.weight"] = _uniform("output.weight", (V, D), D, seed)
    return sd


def mixtral_state_dict(args: dict, seed: int = 0, perturb_norm: bool = True, gain: float = 1.0):
    """Mixtral base-MoE keys (mixtral.py:238-241): all experts of all ranks (master)."""
    D, L, H = args["dim"], args["n_layers"], args["n_heads"]
    Hkv = args.get("n_kv_heads") or H
    hd = D // H  # mixtral.py:65 derives head_dim = dim // n_heads and ignores ModelArgs.head_dim
    V, F = args["vocab_size"], args["hidden_dim"]
    E = args["moe"]["num_experts"]
    sd = {"tok_embeddings.weight": _uniform("tok_embeddings.weight", (V, D), D, seed)}
    for i in range(L):
        p = f"layers.{i}."
        sd[p + "attention.wq.weight"] = _uniform(p + "wq", (H * hd, D), D, seed, gain)
        sd[p + "attention.wk.weight"] = _uniform(p + "wk", (Hkv * hd, D), D, seed, gain)
        sd[p + "attention.wv.weight"] = _uniform(p + "wv", (Hkv * hd, D), D, seed, gain)
        sd[p + "attention.wo.weight"] = _uniform(p + "wo", (D, H * hd), H * hd, seed, gain)
        # a wider router init than 1/sqrt(D) so that top-2 choices are not all near-ties
        sd[p + "feed_forward.gate.weight"] = _uniform(p + "gate", (E, D), D, seed, 4.0)
        for e in range(E):
            q = p + f"feed_forward.experts.{e}."
            sd[q + "w1.weight"] = _uniform(q + "w1", (F, D), D, seed, gain)
            sd[q + "w2.weight"] = _uniform(q + "w2", (D, F), F, seed, gain)
            sd[q + "w3.weight"] = _uniform(q + "w3", (F, D), D, seed, gain)
        sd[p + "attention_norm.weight"] = _norm_weight(p + "an", D, seed, perturb_norm)
        sd[p + "ffn_norm.weight"] = _norm_weight(p + "fn", D, seed, perturb_norm)
    sd["norm.weight"] = _norm_weight("norm", D, seed, perturb_norm)
    sd["output.weight"] = _uniform("output.weight", (V, D), D, seed)
    return sd


def synthetic_tokens(bsz, seqlen, vocab, seed=1234):
    """ids ~ randint(1, vocab): 0 is the pad/ignore id (meta.py:60,419)."""
    g = torch.Generator()
    g.manual_seed(seed)
    return torch.randint(1, vocab, (bsz, seqlen), generator=g, dtype=torch.int64)


# --- tensor-parallel sharding of a master state dict (tensor_parallel.py:34-38) -------------
_COL = ("attention.wq.weight", "attention.wk.weight", "attention.wv.weight",
        "feed_forward.w1.weight", "feed_forward.w3.weight", "output.weight")
_ROW = ("attention.wo.weight", "feed_forward.w2.weight")


def shard_state_dict(sd: dict, rank: int, world: int, kind: str = "llama"):
    """ColumnParallel: dim 0; RowParallel: dim 1; ParallelEmbedding: dim 1;
    Mixtral experts: whole experts [E/world*rank, E/world*(rank+1)) (mixtral.py:237);
    norms and the router gate replicated."""
    if world == 1:
        return dict(sd)
    out = {}
    n_exp = None
    if kind == "mixtral":
        n_exp = 1 + max(int(k.split(".experts.")[1].split(".")[0]) for k in sd if ".experts." in k)
        per = n_exp // world
    for k, v in sd.items():
        if ".experts." in k:
            e = int(k.split(".experts.")[1].split(".")[0])
            if per * rank <= e < per * (rank + 1):
                out[k] = v
        elif k.endswith(_COL):
            out[k] = v.chunk(world, dim=0)[rank].contiguous()
        elif k.endswith(_ROW) or k == "tok_embeddings.weight":
            out[k] = v.chunk(world, dim=1)[rank].contiguous()
        else:
            out[k] = v
    return out


def tensor_digest(t: torch.Tensor) -> dict:
    """dtype, shape and sha256 of the bytes: a stored stand-in for a tensor that a test compares with torch.equal."""
    raw = t.detach().cpu().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes()
    return {"dtype": str(t.dtype), "shape": list(t.shape), "sha256": hashlib.sha256(raw).hexdigest()}
