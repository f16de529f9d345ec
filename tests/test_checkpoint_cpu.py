"""CPU: the on-disk formats either side of the decode path (SURVEY.md 8f rank 1).

* the reference's tensor-parallel checkpoint folders (util/tensor_parallel.py) are read back, merged and
  re-split exactly as the reference shards its layers (oracle.weights.shard_state_dict is the checker);
* an OmniQuant fake-quantised fp16 state dict (oracle.omniquant) is inverted to integers that reproduce it
  bit-exactly;
* the engine's packed shards survive a save / load round trip, and one call turns a checkpoint folder into an
  engine whose weights dequantise to the checkpoint.
"""
import json
import os

import numpy as np
import pytest
import torch

import llama2_accessory_b200 as pkg
from llama2_accessory_b200 import checkpoint as ck
from llama2_accessory_b200 import quant
from llama2_accessory_b200.engine import DecodeEngine, EngineConfig
from oracle import cases, omniquant
from oracle.weights import shard_state_dict, tensor_digest


@pytest.fixture(scope="module", autouse=True)
def _built():
    pkg.build()


def _master(kind):
    args = cases.TINY_LLAMA if kind == "llama" else cases.TINY_MIXTRAL
    return args, cases.master_state_dict(kind, args, seed=3)


def _eq(a, b):
    assert set(a) == set(b), (sorted(set(a) ^ set(b))[:5])
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("kind", ["llama", "mixtral"])
@pytest.mark.parametrize("fmt", ["consolidated", "meta_ori"])
def test_formats_round_trip_and_resharding(tmp_path, kind, fmt):
    args, sd = _master(kind)
    d = str(tmp_path / "ckpt")
    ck.save_tensor_parallel_shards(sd, d, 2, fmt)
    assert ck.infer_checkpoint_format_and_mp_size(d) == (fmt, 2)
    # every stored rank equals the reference's sharding of the master weights
    for r in range(2):
        stored = ck.load_tensor_parallel_shard_state_dict(d, fmt, r, 2)
        assert all(k.startswith("llma.") for k in stored)
        _eq({k[5:]: v for k, v in stored.items()}, shard_state_dict(sd, r, 2, kind))
    # merge 2 -> 1, identity 2 -> 2, split 2 -> 4
    _eq(ck.load_tensor_parallel_state_dict_list(d, 0, 1), sd)
    for r in range(2):
        _eq(ck.load_tensor_parallel_state_dict_list(d, r, 2), shard_state_dict(sd, r, 2, kind))
    for r in range(4):
        _eq(ck.load_tensor_parallel_state_dict_list(d, r, 4), shard_state_dict(sd, r, 4, kind))


def test_split_of_a_single_file_checkpoint_and_model_wrapper(tmp_path):
    args, sd = _master("llama")
    d = str(tmp_path / "one")
    ck.save_tensor_parallel_shards(sd, d, 1, "consolidated", wrap_model=True)
    assert isinstance(torch.load(os.path.join(d, "consolidated.00-of-01.model.pth"))["model"], dict)
    for r in range(2):
        _eq(ck.load_tensor_parallel_state_dict_list(d, r, 2), shard_state_dict(sd, r, 2, "llama"))
    d2 = str(tmp_path / "bare")
    ck.save_tensor_parallel_shards(sd, d2, 1, "consolidated", wrap_model=False)
    _eq(ck.load_tensor_parallel_state_dict_list(d2), sd)


def test_diff_checkpoint_is_added_and_base_overrides(tmp_path):
    args, sd = _master("llama")
    base, diff, base2 = str(tmp_path / "base"), str(tmp_path / "diff"), str(tmp_path / "base2")
    ck.save_tensor_parallel_shards(sd, base, 2, "consolidated")
    delta = {k: torch.full_like(v, 0.125) for k, v in sd.items() if "attention.wq" in k or k == "norm.weight"}
    ck.save_tensor_parallel_shards(delta, diff, 2, "consolidated_diff")
    assert ck.infer_checkpoint_format_and_mp_size(diff) == ("consolidated_diff", 2)
    got = ck.load_tensor_parallel_state_dict_list([base, diff])
    for k, v in sd.items():
        assert torch.equal(got[k], v + delta[k] if k in delta else v), k
    # a later full checkpoint overrides what came before
    other = {k: v * 2 for k, v in sd.items() if "feed_forward.w2" in k}
    ck.save_tensor_parallel_shards(other, base2, 1, "consolidated")
    got = ck.load_tensor_parallel_state_dict_list([base, diff, base2])
    for k in other:
        assert torch.equal(got[k], other[k])
    with pytest.raises(AssertionError):
        ck.load_tensor_parallel_state_dict_list([diff, base])


def test_format_inference_failures_match_the_reference(tmp_path):
    args, sd = _master("llama")
    with pytest.raises(NotImplementedError):
        ck.infer_checkpoint_format_and_mp_size(str(tmp_path / "nope"))
    empty = tmp_path / "empty"
    empty.mkdir()
    (empty / "readme.txt").write_text("x")
    with pytest.raises(NotImplementedError, match="do not match"):
        ck.infer_checkpoint_format_and_mp_size(str(empty))
    d = str(tmp_path / "mixed")
    ck.save_tensor_parallel_shards(sd, d, 1, "consolidated")
    ck.save_tensor_parallel_shards(sd, d, 1, "meta_ori")
    with pytest.raises(NotImplementedError, match="Multiple matched format"):
        ck.infer_checkpoint_format_and_mp_size(d)
    d = str(tmp_path / "hole")
    ck.save_tensor_parallel_shards(sd, d, 4, "consolidated")
    os.remove(os.path.join(d, "consolidated.01-of-04.model.pth"))
    with pytest.raises(NotImplementedError, match="expected file"):
        ck.infer_checkpoint_format_and_mp_size(d)
    d = str(tmp_path / "three")
    ck.save_tensor_parallel_shards({k: v for k, v in sd.items() if "norm" in k}, d, 3, "consolidated")
    with pytest.raises(NotImplementedError, match="redistribute"):
        ck.load_tensor_parallel_state_dict(d, 0, 2)


def test_meta_config_and_tokenizer_probing(tmp_path):
    d = tmp_path / "m"
    d.mkdir()
    with pytest.raises(ValueError, match="llama_type"):
        ck.read_model_meta(str(d))
    (d / "meta.json").write_text(json.dumps({"llama_type": "llama"}))
    m = ck.read_model_meta(str(d))
    assert m == {"llama_type": "llama", "config": {}, "tokenizer_path": None}
    (d / "config.json").write_text(json.dumps({"dim": 512, "n_heads": 4}))
    extra = tmp_path / "extra.json"
    extra.write_text(json.dumps({"n_heads": 8, "rope_theta": 5e5}))
    assert ck.read_model_meta(str(d))["config"] == {"dim": 512, "n_heads": 4}
    assert ck.read_model_meta([str(tmp_path), str(d)], llama_config=[str(d / "config.json"), str(extra)])["config"] == {
        "dim": 512, "n_heads": 8, "rope_theta": 5e5}
    (d / "tokenizer.json").write_text("{}")
    assert ck.probe_tokenizer_path_from_pretrained(str(d)) is None  # needs tokenizer_config.json too
    (d / "tokenizer_config.json").write_text("{}")
    assert ck.probe_tokenizer_path_from_pretrained(str(d)) == str(d)
    (d / "tokenizer.model").write_bytes(b"spm")
    assert ck.probe_tokenizer_path_from_pretrained(str(d)) == str(d / "tokenizer.model")


@pytest.mark.parametrize("bits,gs", [(4, 0), (4, 128), (4, 64), (3, 0), (3, 128), (2, 64), (2, 128)])
def test_fake_quantised_weights_are_inverted_bit_exactly(bits, gs):
    g = torch.Generator().manual_seed(bits * 100 + gs)
    w = ((torch.rand(96, 512, generator=g) * 2 - 1) / 512 ** 0.5).half()
    w[5] = w[5].abs()          # a row without negative values (zero point 0)
    w[6] = -w[6].abs() - 0.01  # all negative: zero point beyond the top level
    rec = omniquant.quantize_weight(w, bits, gs)
    fake = omniquant.dequantize(rec["q"], rec["scale"].float(), rec["zero"].float(), rec["group_size"]).half()
    q, s, z, gg = ck.recover_quant_from_fake(fake, bits, gs)
    assert gg == rec["group_size"] and int(q.max()) <= 2 ** bits - 1
    assert torch.equal(quant.dequantize(q, s, z, gg), fake)
    # what is observable is recovered exactly: the level index q - z wherever the stored scale was recovered as is
    same = (s == rec["scale"].half()).reshape(96, -1, 1).expand(-1, -1, gg).reshape(96, 512)
    n_rec = q.float() - z.float().repeat_interleave(gg, dim=1)
    n_ref = rec["q"].float() - rec["zero"].float().repeat_interleave(gg, dim=1)
    assert float(same.float().mean()) > 0.9
    assert torch.equal(n_rec[same], n_ref[same])


def test_recovery_rejects_weights_that_are_not_on_a_grid():
    w = torch.randn(16, 256).half()
    with pytest.raises(ValueError):
        ck.recover_quant_from_fake(w, 4, 0)
    # a genuine W4 checkpoint is not a W2 checkpoint
    rec = omniquant.quantize_weight(w, 4, 128)
    fake = omniquant.dequantize(rec["q"], rec["scale"].float(), rec["zero"].float(), 128).half()
    with pytest.raises(ValueError):
        ck.recover_quant_from_fake(fake, 2, 128)


def _dequant_packed_fp16(pl):
    q = quant.unpack_quantized(pl)
    sz = torch.from_numpy(pl.scales.cpu().numpy().view(np.float16).copy())
    N, K = pl.N, pl.K
    if pl.group_size == 0:
        sz = sz.reshape(N, 2)
        return quant.dequantize(q, sz[:, 0:1].contiguous(), sz[:, 1:2].contiguous(), K)
    G = K // pl.group_size
    sz = sz.reshape(N // 16, G, 16, 2).permute(0, 2, 1, 3).reshape(N, G, 2)
    return quant.dequantize(q, sz[..., 0].contiguous(), sz[..., 1].contiguous(), pl.group_size)


@pytest.mark.parametrize("kind,bits,gs", [("llama", 4, 0), ("llama", 4, 128), ("mixtral", 4, 0)])
def test_checkpoint_folder_to_engine_and_packed_round_trip(tmp_path, kind, bits, gs):
    args, sd = _master(kind)
    sd_fake, recs = omniquant.fake_quantize_state_dict(sd, bits, gs)
    d = str(tmp_path / "omni")
    ck.save_tensor_parallel_shards(sd_fake, d, 2, "consolidated")
    with open(os.path.join(d, "meta.json"), "w") as f:
        json.dump({"llama_type": kind}, f)
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump({k: v for k, v in args.items() if k not in ("max_seq_len", "max_batch_size")}, f)
    eng, meta = ck.build_engine_from_pretrained(d, bits=bits, group_size=gs, fake_quantised=True, max_seq_len=64,
                                                max_batch_size=4, device="cpu")
    assert meta["llama_type"] == kind and eng.cfg.dim == args["dim"]
    # the packed weights dequantise to the checkpoint's fp16 values, bit for bit
    lw = eng.layers[1]
    wo = _dequant_packed_fp16(lw.wo)
    assert torch.equal(wo, sd_fake["layers.1.attention.wo.weight"])
    qkv = _dequant_packed_fp16(lw.wqkv)
    ref = torch.cat([sd_fake[f"layers.1.attention.{n}.weight"] for n in ("wq", "wk", "wv")], 0)
    assert torch.equal(qkv, ref)
    assert torch.equal(eng.tok_emb, sd_fake["tok_embeddings.weight"])
    # packed shards: save, load into a fresh engine, identical device images
    out = str(tmp_path / "packed")
    fn = ck.save_packed(eng, out)
    assert os.path.basename(fn) == "b200_packed.00-of-01.pth"
    eng2 = DecodeEngine(eng.cfg, "cpu")
    ck.load_packed(eng2, out)
    assert torch.equal(eng2.tok_emb, eng.tok_emb) and torch.equal(eng2.lm_head.qweight, eng.lm_head.qweight)
    for a, b in zip(eng.layers, eng2.layers):
        for name in ("wqkv", "wo", "w13", "w2"):
            pa, pb = getattr(a, name), getattr(b, name)
            assert (pa is None) == (pb is None)
            if pa is not None:
                assert torch.equal(pa.qweight, pb.qweight) and torch.equal(pa.scales, pb.scales)
                assert (pa.bits, pa.N, pa.K, pa.group_size) == (pb.bits, pb.N, pb.K, pb.group_size)
        assert len(a.e_w13) == len(b.e_w13)
        for pa, pb in zip(a.e_w13 + a.e_w2, b.e_w13 + b.e_w2):
            assert torch.equal(pa.qweight, pb.qweight) and torch.equal(pa.scales, pb.scales)
    # a shard written for another configuration is refused
    other = EngineConfig.from_model_args(kind, dict(args, max_seq_len=64), bits=bits, group_size=gs, tp_rank=0, tp_world=1)
    other.bits = 3 if bits == 4 else 4
    with pytest.raises(ValueError, match="bits"):
        ck.load_packed(DecodeEngine(other, "cpu"), out)


def test_merge_and_inference_agree_with_the_reference_loader(tmp_path):
    """The UNMODIFIED accessory/util/tensor_parallel.py read the same folders (tests/golden/reference_tp_loader.json, made
    by oracle/make_golden_loader.py): format inference, shard file names and the merged TP = 1 state dict must agree tensor
    for tensor, the merged dict must fit the reference Transformer's parameter names, and the same malformed folders are
    refused."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tp_loader.json")) as f:
        gold = json.load(f)
    args, sd = _master("llama")
    ref_keys = set(gold["model_keys"])
    for fmt, g in gold["formats"].items():
        d = str(tmp_path / fmt)
        ck.save_tensor_parallel_shards(sd, d, 2, fmt)
        assert ck.infer_checkpoint_format_and_mp_size(d) == tuple(g["inferred"]) == (fmt, 2)
        assert ck.get_tensor_parallel_shards_file_name(fmt, 2) == g["shard_file_names"]
        mine = ck.load_tensor_parallel_state_dict(d, 0, 1, fmt)
        assert set(g["merged"]) == set(mine)
        for k in mine:
            assert tensor_digest(mine[k]) == g["merged"][k], k
        # and it loads into the reference model without missing / unexpected weights
        assert set(mine) <= ref_keys and all("clip" in k or "rope" in k or "freqs" in k for k in ref_keys - set(mine))
    assert gold["refused"] == {"empty": "NotImplementedError", "mixed": "NotImplementedError"}
    for bad in gold["refused"]:
        d = tmp_path / bad
        d.mkdir()
        if bad == "mixed":
            ck.save_tensor_parallel_shards(sd, str(d), 1, "consolidated")
            ck.save_tensor_parallel_shards(sd, str(d), 1, "meta_ori")
        else:
            (d / "x.txt").write_text("x")
        with pytest.raises(NotImplementedError):
            ck.infer_checkpoint_format_and_mp_size(str(d))


def test_every_tensor_parallel_rank_packs_its_slice_of_the_master_quantisation(tmp_path):
    """quantise the MASTER weights, then shard (SURVEY.md 8e): the ranks of a TP = 2 engine built from one folder hold
    row / column slices of the SAME integers and scales as the TP = 1 engine, and save one packed file each."""
    args, sd = _master("llama")
    sd_fake, _ = omniquant.fake_quantize_state_dict(sd, 4, 128)
    d = str(tmp_path / "ckpt")
    ck.save_tensor_parallel_shards(sd_fake, d, 1, "consolidated")
    with open(os.path.join(d, "meta.json"), "w") as f:
        json.dump({"llama_type": "llama"}, f)
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump({k: v for k, v in args.items() if k not in ("max_seq_len", "max_batch_size")}, f)
    kw = dict(bits=4, group_size=128, fake_quantised=True, max_seq_len=64, max_batch_size=4, device="cpu")
    full, _ = ck.build_engine_from_pretrained(d, **kw)
    wo_full = _dequant_packed_fp16(full.layers[0].wo)
    w2_full = _dequant_packed_fp16(full.layers[0].w2)
    out = str(tmp_path / "packed")
    for r in range(2):
        eng, _ = ck.build_engine_from_pretrained(d, tp_rank=r, tp_world=2, **kw)
        assert torch.equal(_dequant_packed_fp16(eng.layers[0].wo), wo_full.chunk(2, dim=1)[r])      # row-parallel: K slice
        assert torch.equal(_dequant_packed_fp16(eng.layers[0].w2)[:, :eng.F_raw], w2_full.chunk(2, dim=1)[r])
        q = _dequant_packed_fp16(eng.layers[0].wqkv)                                                 # column-parallel: head rows
        assert torch.equal(q[:eng.Hq * 128], sd_fake["layers.0.attention.wq.weight"].chunk(2, dim=0)[r])
        assert eng.lm_head.N == args["vocab_size"] // 2
        assert os.path.basename(ck.save_packed(eng, out)) == f"b200_packed.{r:02d}-of-02.pth"
        again = DecodeEngine(eng.cfg, "cpu")
        ck.load_packed(again, out)
        assert torch.equal(again.layers[1].w13.qweight, eng.layers[1].w13.qweight)


@pytest.mark.parametrize("kind,fmt", [("llama", "consolidated"), ("llama", "meta_ori"), ("mixtral", "consolidated")])
def test_lazy_merged_state_dict_equals_the_eager_loader(tmp_path, kind, fmt):
    """Streaming loader (one merged tensor materialised per lookup over memory-mapped shards) vs the eager merge: same keys in
    the same order, same values -- at TP = 1 from a 4-way folder and as rank 1 of 2."""
    args, sd = _master(kind)
    d = str(tmp_path / "ck")
    ck.save_tensor_parallel_shards(sd, d, 4, fmt)
    for tp_rank, tp_world in ((0, 1), (1, 2)):
        eager = ck.load_tensor_parallel_state_dict_list([d], tp_rank, tp_world)
        lazy = ck.LazyMergedStateDict(d, tp_rank, tp_world)
        assert list(lazy) == list(eager) and len(lazy) == len(eager)
        for k in eager:
            assert k in lazy and torch.equal(lazy[k], eager[k]), k
        assert "not.a.key" not in lazy
    with pytest.raises(NotImplementedError):
        ck.LazyMergedStateDict(d, 0, 8)  # the split direction stays with the eager loader


def test_streaming_engine_build_equals_the_eager_build(tmp_path):
    """build_engine_from_pretrained on one folder streams (LazyMergedStateDict + LazyQuantRecords); a two-entry path list
    (base + diff of zeros) takes the eager route: identical packed images."""
    args, sd = _master("llama")
    sd_fake, recs = omniquant.fake_quantize_state_dict(sd, 4, 128)
    d = str(tmp_path / "omni")
    ck.save_tensor_parallel_shards(sd_fake, d, 2, "consolidated")
    z = str(tmp_path / "zero_diff")
    ck.save_tensor_parallel_shards({k: torch.zeros_like(v) for k, v in sd_fake.items()}, z, 2, "consolidated_diff")
    for p in (d, z):
        with open(os.path.join(p, "meta.json"), "w") as f:
            json.dump({"llama_type": "llama"}, f)
        with open(os.path.join(p, "config.json"), "w") as f:
            json.dump({k: v for k, v in args.items() if k not in ("max_seq_len", "max_batch_size")}, f)
    kw = dict(bits=4, group_size=128, fake_quantised=True, max_seq_len=64, max_batch_size=4, device="cpu")
    a, _ = ck.build_engine_from_pretrained(d, **kw)
    b, _ = ck.build_engine_from_pretrained([d, z], **kw)
    lz = ck.LazyQuantRecords(ck.LazyMergedStateDict(d), 4, 128)
    assert set(lz) == set(recs) and "norm.weight" not in lz
    k0 = "layers.0.attention.wq.weight"
    assert torch.equal(lz[k0]["q"], recs[k0]["q"]) and torch.equal(lz[k0]["scale"], recs[k0]["scale"])
    assert torch.equal(a.tok_emb, b.tok_emb) and torch.equal(a.lm_head.qweight, b.lm_head.qweight)
    for la, lb in zip(a.layers, b.layers):
        for name in ("wqkv", "wo", "w13", "w2"):
            pa, pb = getattr(la, name), getattr(lb, name)
            assert torch.equal(pa.qweight, pb.qweight) and torch.equal(pa.scales, pb.scales), name
