"""Per-CTA %globaltimer stamps of the five launches of one layer (+ the next layer's QKV) inside the graph-replayed bs = 1
decode step (LLaMA2-7B W4 ctx 2048): where CTAs start relative to each other, when the dependency resolves, when x is
staged, when the first weight slot is consumed, when the MMA loop and the epilogue end."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np
import torch
import llama2_accessory_b200 as pkg
pkg.build()
from llama2_accessory_b200 import _cabi
from llama2_accessory_b200.engine import DecodeEngine, EngineConfig

MODEL = dict(dim=4096, n_layers=32, n_heads=32, n_kv_heads=None, multiple_of=256, ffn_dim_multiplier=None,
             norm_eps=1e-5, rope_theta=10000.0, vocab_size=32000, max_seq_len=2048 + 352)
CTX, BSZ, LAYER = 2048, 1, int(os.environ.get("LAYER", "15"))
lib = _cabi.lib()
KNOB_SETS = [ks for ks in os.environ.get("KNOBS", "").split(";")] or [""]
ALL_KNOBS = set()
for ks in KNOB_SETS:
    for kv in ks.split(","):
        if "=" in kv:
            ALL_KNOBS.add(kv.split("=")[0])
eng = DecodeEngine(EngineConfig.from_model_args("llama", MODEL, bits=4, group_size=0), "cuda")
eng.load_random(0)
eng.allocate_kv_cache(BSZ)
eng.fill_kv_cache_noise()
NROW, NCTA, NL = 400, 320, 6
tl = torch.zeros((NROW, 8), dtype=torch.int64, device="cuda")
tlc = torch.zeros((NL, NCTA, 16), dtype=torch.int64, device="cuda")
def run(ks):
    for k in ALL_KNOBS:
        lib.b200_tune(k.encode(), -1)
    defaults = {"B200_PF_KB": 96, "B200_PF_KV": 1, "B200_G1_ARED": 1, "B200_KEEP_CONST": 1, "B200_CONST_PF": 1, "B200_ATTN_EVEN": 1}
    for k in ALL_KNOBS:
        if k in defaults:
            lib.b200_tune(k.encode(), defaults[k])
    for kv in ks.split(","):
        if "=" in kv:
            k, v = kv.split("=")
            lib.b200_tune(k.encode(), int(v))
    eng._graphs.clear()
    print(f"######## knobs: {ks or '(defaults)'}")
    eng.tokens[:BSZ].fill_(5); eng.pos[:BSZ].fill_(CTX)
    eng._step(BSZ, 1, eng.cache_seq); torch.cuda.synchronize()
    lib.b200_timeline(C.c_void_p(tl.data_ptr()), NROW)
    lib.b200_timeline_cta(C.c_void_p(tlc.data_ptr()), 161 + 5 * LAYER, NL, NCTA)   # rows 0..160: the eager warm-up pass of the capture
    g, n = eng.capture_greedy_loop(BSZ)
    lib.b200_timeline(None, 0)
    lib.b200_timeline_cta(None, 0, 0, 0)
    eng.tokens[:BSZ].fill_(1234); eng.pos[:BSZ].fill_(CTX)
    for _ in range(30):
        g.replay()
    torch.cuda.synchronize()
    tl.zero_(); tl[:, 0] = torch.iinfo(torch.int64).max; tlc.zero_()
    g.replay(); torch.cuda.synchronize()
    t = tlc.cpu().numpy().astype(np.float64)
    names = ["qkv", "attn", "wo", "w13", "w2", "qkv+1"]
    cols = [(0, "start"), (4, "dep"), (8, "x-loads"), (9, "normbar"), (1, "xstage"), (7, "slot0"), (2, "mmaend"), (6, "epi0"), (3, "end")]
    t0 = t[0][:, 0][t[0][:, 0] > 0].min()
    print(f"per-CTA stamps, us relative to the first CTA start of layer {LAYER}'s QKV; min / p10 / median / p90 / max over CTAs")
    for li in range(NL):
        r = t[li]
        live = r[:, 0] > 0
        r = r[live]
        print(f"== {names[li]}: {len(r)} CTAs; work units/CTA histogram {dict(zip(*[x.tolist() for x in np.unique(r[:, 5], return_counts=True)]))}")
        for c, nm in cols:
            v = r[:, c][r[:, c] > 0]
            if len(v) == 0:
                continue
            v = (v - t0) / 1000.0
            print(f"   {nm:7s} n={len(v):3d}  {v.min():7.2f} {np.percentile(v, 10):7.2f} {np.median(v):7.2f} {np.percentile(v, 90):7.2f} {v.max():7.2f}")
        # per-CTA durations: start -> end, grouped by work units
        for u in np.unique(r[:, 5]):
            sel = r[r[:, 5] == u]
            ok = (sel[:, 3] > 0) & (sel[:, 0] > 0)
            if ok.sum():
                d = (sel[ok, 3] - sel[ok, 0]) / 1000.0
                s = (sel[ok, 0] - t0) / 1000.0
                print(f"   units={int(u)}: n={int(ok.sum())} start median {np.median(s):.2f}  life (start->end) median {np.median(d):.2f} max {d.max():.2f}")
    

for ks in KNOB_SETS:
    run(ks)
