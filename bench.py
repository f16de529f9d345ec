#!/usr/bin/env python
"""bench.py -- decode tokens/s of the B200 quantised-decode engine on BASELINE.json's headline workload:
LLaMA2-7B OmniQuant W4A16 (per-channel), bs=1, ctx=2048, synthetic random-init weights and prompts.

    python bench.py --gpus N --steps K --warmup W           (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                    (the reference path's CPU implementation)

One "step" = one decode step (one token for the whole batch) through all 32 layers + lm_head.
  value      device-resident: tokens stay on the GPU (step -> argmax -> next step) in one CUDA graph;
             timed with CUDA events over exactly K steps, barrier + synchronize on both sides, max over ranks.
  e2e        the same K steps through the public drop-in API (Transformer.forward_inference): every step
             copies the token from pinned host memory, and reads the sampled token back to the host.
  roofline   the dequant-GEMV kernel (the only kernel that touches weights): algorithmic packed bytes of
             the 4 GEMVs of every layer / CUDA-event time of running just those launches, vs MEASURED_PEAKS.
  cpu_baseline  the reference's own llama.py forward_inference (staged unmodified under oracle/_ref) on the host
             cores: real full-depth decode steps, as many as fit a 25 s box.  Host threads = the fastest count of a short
             sweep up to the CPUs the process may use (affinity mask capped by the cgroup quota), see calibrate_threads.
N GPUs = tensor parallel over N ranks (the reference's scheme; strong scaling: one model, one token stream).

--dump-outputs DIR writes what the last timed step of `value` computed, as a caller of that step receives it:
  DIR/logits.npy      float32 [bsz, vocab]   the step's logits
  DIR/next_token.npy  float64 [bsz]          the greedy token the step fed back (argmax of those logits)
Weights, KV cache and the first token are drawn from fixed seeds, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CTX = 2048
BSZ = 1
MODEL = dict(dim=4096, n_layers=32, n_heads=32, n_kv_heads=None, multiple_of=256, ffn_dim_multiplier=None,
             norm_eps=1e-5, rope_theta=10000.0, vocab_size=32000)
WORKLOAD = "LLaMA2-7B OmniQuant W4A16 (per-channel) decode bs=1 ctx=2048"


def _log(msg):
    if os.environ.get("B200_BENCH_VERBOSE"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def _finish(world):
    """Multi-rank exit: NCCL communicators referenced by captured CUDA graphs can make destroy_process_group() hang;
    synchronise, flush and leave with status 0."""
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture summary of this round (profiles/r02_ncu_traffic.json: {kernel substring: bytes}); None when not captured."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    try:
        d = json.load(open(p))
        for k, v in d.items():
            if k in kernel_name:
                return float(v)
    except Exception:
        pass
    return None


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path on the host cores (bounded sample)
# ---------------------------------------------------------------------------------------------------
METRIC = "decode tokens/s (LLaMA2-7B W4A16 bs=1; p50 per-token ms in config)"


def host_threads():
    """CPUs this process may use: the affinity mask, capped by the cgroup CPU quota (a container that SEES 128 CPUs may be
    allowed the time of 16: an OpenMP team of 128 then spends its life in barrier spins)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:  # cgroup v2: "<quota|max> <period>"
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = int(q) / int(per)
    except (OSError, ValueError):
        pass
    if quota is None:
        try:  # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def calibrate_threads(limit):
    """The host thread count the reference's CPU forward is timed with = the fastest of a short sweep over a
    memory-bound fp32 linear at M = 1 (the shape of a decode step's work: [1, 8192] x [8192, 8192], 256 MB of weights,
    larger than any cache), not simply every CPU the process can see.  On the 1-GPU boxes of round 1 / 2 "all 128
    visible CPUs" ran the very same forward 47x slower than 8 threads of the build container (17 s vs 0.36 s per step):
    an oversubscribed OpenMP team.  Ascending order, so the pool never holds more threads than were tried; a count must
    be 3 % faster to replace a smaller one; the sweep stops once a count is 3x slower than the best so far.
    -> (threads, {count: ms per linear})"""
    import torch
    import torch.nn.functional as F
    cands = sorted({c for c in (2, 4, 8, 12, 16, 24, 32, 48, 64, 96, 128, 192, 256, limit) if 1 <= c <= limit} | {min(limit, 1)})
    torch.set_num_threads(cands[0])
    g = torch.Generator().manual_seed(0)
    W = torch.rand((8192, 8192), generator=g) - 0.5
    x = torch.rand((1, 8192), generator=g) - 0.5
    best, best_t, tried = cands[0], float("inf"), {}
    with torch.inference_mode():
        for c in cands:
            torch.set_num_threads(c)
            F.linear(x, W)  # first parallel region at this team size (thread creation)
            reps = 5
            t0 = time.perf_counter()
            for _ in range(reps):
                F.linear(x, W)
            dt = (time.perf_counter() - t0) / reps
            tried[c] = round(1000.0 * dt, 3)
            if dt < 0.97 * best_t:
                best, best_t = c, dt
            elif dt > 3.0 * best_t:
                break
    torch.set_num_threads(best)
    return best, tried


class CpuReference:
    """The reference's decode step on the host: the UNMODIFIED accessory/model/LLM/llama.py Transformer
    (oracle/_ref staged copy on the GPU box, /root/reference in the build container; the bit-pinned port only if
    neither exists), all 32 blocks, OmniQuant fake-quantised W4 weights (fp16 values) computed in fp32, KV cache
    pre-filled to ctx 2048.  One step = one real Transformer.forward_inference(tokens[1,1], start_pos) call."""

    def __init__(self, bits=4, group_size=0):
        import torch
        from oracle import big_model
        self.torch = torch
        self.visible = host_threads()
        self.threads, self.thread_sweep = calibrate_threads(self.visible)
        t0 = time.perf_counter()
        args = dict(MODEL, max_seq_len=CTX + 64, max_batch_size=BSZ)
        # weight preparation (random draw + quantiser) runs on the GPU when there is one: it is not what is timed
        self.model, self.kind, _ = big_model.build(args, bits=bits, group_size=group_size, dtype=torch.float32,
                                                   device="cpu", fast=True)
        big_model.fill_kv_noise(self.model, BSZ)
        g = torch.Generator().manual_seed(1234)
        self.tok = torch.randint(1, MODEL["vocab_size"], (BSZ, 1), generator=g)
        self.prep_s = time.perf_counter() - t0
        self.pos = CTX

    def step(self):
        t0 = time.perf_counter()
        with self.torch.inference_mode():
            logits = self.model.forward_inference(self.tok, self.pos)
            self.tok = logits.argmax(dim=-1, keepdim=True)
        self.pos = CTX + (self.pos + 1 - CTX) % 32
        return time.perf_counter() - t0

    def describe(self):
        src = ("unmodified reference llama.py Transformer.forward_inference" if self.kind == "reference"
               else "oracle port of llama.py forward_inference")
        return (f"{src}, all 32 blocks + lm_head, OmniQuant fake-quantised W4 weights computed in fp32, "
                f"one decode step at ctx 2048 per timed step, {self.threads} host threads (fastest of a sweep up to the "
                f"{self.visible} CPUs the process may use)")


def cpu_decode_sample(budget_s=25.0, max_steps=8):
    """cpu_baseline leg of the product arm: real full-depth decode steps of the reference on the host, as many as fit
    in `budget_s` (at least one after one warm-up)."""
    ref = CpuReference()
    ref.step()  # warm-up (page faults, thread pool)
    ts, t_all = [], time.perf_counter()
    while len(ts) < max_steps and (not ts or time.perf_counter() - t_all + ts[-1] < budget_s):
        ts.append(ref.step())
    med = statistics.median(ts)
    return BSZ / med, {"kind": ref.kind, "cores": ref.threads, "cpus_usable": ref.visible, "thread_sweep_ms": ref.thread_sweep,
                       "steps_timed": len(ts), "step_s": med, "prep_s": ref.prep_s, "sample": ref.describe()}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, all host threads; rank 0 only.
    Every timed step is one real full-depth decode step; when the host is too slow for `--steps` of them inside the
    time box, fewer are run and `steps` reports the number actually timed (no extrapolation)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all0 = time.perf_counter()
    ref = CpuReference(bits=args.bits, group_size=args.group_size)
    budget = float(os.environ.get("B200_REF_BUDGET_S", "150"))
    t_first = ref.step()  # first warm-up step
    W = 1
    while W < min(args.warmup, 3) and (W + 1) * t_first < 0.2 * budget:
        ref.step()
        W += 1
    ts = []
    t0 = time.perf_counter()
    while len(ts) < args.steps and (not ts or (time.perf_counter() - t0) + max(ts) < budget):
        ts.append(ref.step())
    total = sum(ts)
    K = len(ts)
    v = BSZ * K / total
    ts.sort()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": K, "warmup": W, "steps_requested": args.steps, "ms_per_step": 1000.0 * total / K,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "bits": args.bits, "group_size": args.group_size, "bsz": BSZ, "ctx": CTX,
                   "parallelism": "cpu", "p50_ms_per_token": 1000.0 * ts[K // 2],
                   "note": "CPU arm: fake-quantised fp16 weight values of the same model, fp32 arithmetic on the host"},
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": ref.threads, "cpus_usable": ref.visible,
                         "thread_sweep_ms": ref.thread_sweep, "kind": ref.kind, "sample": ref.describe()},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "prep_s": ref.prep_s, "wall_s": time.perf_counter() - t_all0,
    }))


def tp_parity_check(rank, world, local, group):
    """bs = 1 prefill 4 + 6 decode steps of a small LLaMA (8 kv heads, so it shards up to TP = 8) on the TP = world engine
    vs a TP = 1 engine run on rank 0's GPU: max |logit difference| (the row-parallel partial sums are added in rank
    order in fp32, so the difference is fp16 rounding of the summed vector)."""
    import torch
    import torch.distributed as dist
    from llama2_accessory_b200.engine import DecodeEngine, EngineConfig, llama_ffn_hidden
    args = dict(dim=1024, n_layers=2, n_heads=8, n_kv_heads=8, multiple_of=256, ffn_dim_multiplier=None, norm_eps=1e-5,
                rope_theta=10000.0, vocab_size=1024, max_seq_len=64, max_batch_size=2)
    # seeded master weights of the small model, identical on every rank (U(+-1/sqrt(fan_in)), norm weights near 1): the
    # product arm generates its own inputs and does not touch oracle/
    g = torch.Generator().manual_seed(3)
    D, V, F = args["dim"], args["vocab_size"], llama_ffn_hidden(args["dim"], args["multiple_of"])

    def uni(n, k):
        return ((torch.rand((n, k), generator=g) * 2 - 1) / k ** 0.5).half()

    def near_one(n):
        return (1.0 + 0.1 * (torch.rand(n, generator=g) * 2 - 1)).half()
    sd = {"tok_embeddings.weight": uni(V, D), "norm.weight": near_one(D), "output.weight": uni(V, D)}
    for i in range(args["n_layers"]):
        p = f"layers.{i}."
        sd.update({p + "attention.wq.weight": uni(D, D), p + "attention.wk.weight": uni(D, D), p + "attention.wv.weight": uni(D, D),
                   p + "attention.wo.weight": uni(D, D), p + "feed_forward.w1.weight": uni(F, D),
                   p + "feed_forward.w2.weight": uni(D, F), p + "feed_forward.w3.weight": uni(F, D),
                   p + "attention_norm.weight": near_one(D), p + "ffn_norm.weight": near_one(D)})
    toks = torch.randint(1, V, (1, 10), generator=torch.Generator().manual_seed(5)).cuda()

    def run(eng):
        outs = [eng.forward_inference(toks[:, :4], 0).float().clone()]
        for j in range(6):
            outs.append(eng.forward_inference(toks[:, 4 + j:5 + j], 4 + j).float().clone())
        return torch.stack(outs)
    eng = DecodeEngine(EngineConfig.from_model_args("llama", args, bits=4, group_size=0, tp_rank=rank, tp_world=world),
                       f"cuda:{local}", group=group)
    eng.load_master_state_dict(sd)
    got = run(eng)
    ar_err = int(eng._ar["step"][1]) if eng._ar is not None else 0
    path = ("persistent dataflow kernel" if (eng.mega_supported(1) and eng.mega_dataflow) else
            "persistent barrier kernel" if eng.mega_supported(1) else "separate kernels + NCCL all-reduce")
    res = torch.zeros(2, device=f"cuda:{local}", dtype=torch.float64)
    if rank == 0:
        e1 = DecodeEngine(EngineConfig.from_model_args("llama", args, bits=4, group_size=0), f"cuda:{local}")
        e1.load_master_state_dict(sd)
        ref = run(e1)
        res[0] = float((got - ref).abs().max())
        res[1] = float(ref.abs().max())
    dist.broadcast(res, src=0)
    same = got.clone()
    dist.broadcast(same, src=0)
    if eng.ar_fused_supported(1) and not eng.mega_supported(1):
        path = "separate kernels, all-reduce fused into the GEMVs (LL push / rank-ordered sum)"
    flag = torch.tensor([float(ar_err)], device=f"cuda:{local}")
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    return {"case": "LLaMA dim 1024 x 2 layers, 8 kv heads, W4 per-channel, bs=1 prefill 4 + 6 decode",
            "max_abs_diff_vs_tp1": float(res[0]), "logits_absmax": float(res[1]),
            "ranks_bit_identical": bool(torch.equal(same, got)), "decode_path": path, "poll_timeouts": int(flag.item())}


def tp_warmup_verdict(tokens, ar_err):
    """Every rank calls this with the tokens it holds after the warm-up steps and its own poll-time-out word; every rank gets
    the SAME answer (same_tokens_on_all_ranks, timeouts_on_any_rank), so that all of them take the same path afterwards."""
    import torch
    import torch.distributed as dist
    tk = tokens.detach().to(torch.float64).reshape(-1)
    lo, hi = tk.clone(), tk.clone()
    bad = torch.tensor([float(ar_err)], device=tokens.device, dtype=torch.float64)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(bad, op=dist.ReduceOp.MAX)
    return bool(torch.equal(lo, hi)), int(bad.item())


def dump_outputs(out_dir, logits, tokens):
    """The last timed step's results as DIR/<name>.npy (float32 / float64: 128 KB at the headline workload)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), logits.float().cpu().numpy())
    np.save(os.path.join(out_dir, "next_token.npy"), tokens.cpu().numpy().astype(np.float64))


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--bits", type=int, default=4)
    ap.add_argument("--group-size", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's logits and next token as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU engine (--impl b200)")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        group = dist.group.WORLD
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    import llama2_accessory_b200 as pkg
    pkg.build()
    from llama2_accessory_b200 import ops
    from llama2_accessory_b200.engine import DecodeEngine, EngineConfig
    from llama2_accessory_b200.model.llama_b200 import Transformer as B200Transformer

    K, W = args.steps, args.warmup
    max_seq = (CTX + 2 * (K + W) + 64 + 31) // 32 * 32
    cfg = EngineConfig.from_model_args("llama", dict(MODEL, max_seq_len=max_seq), bits=args.bits,
                                       group_size=args.group_size, tp_rank=rank, tp_world=world)
    eng = DecodeEngine(cfg, f"cuda:{local}", group=group)
    eng.use_pdl = not args.no_pdl
    eng.load_random(seed=0)
    eng.allocate_kv_cache(BSZ)
    eng.fill_kv_cache_noise(0.5, seed=1)
    dev = eng.device

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- (0) TP > 1: logits of a tiny model at TP = world vs TP = 1 (same kernels, same packed weights) ----------------
    tp_parity = None
    if world > 1:
        tp_parity = tp_parity_check(rank, world, local, group)
        bad = (tp_parity["poll_timeouts"] or not tp_parity["ranks_bit_identical"]
               or not (tp_parity["max_abs_diff_vs_tp1"] <= 8e-3))
        # the verdict must be the SAME on every rank (ranks_bit_identical is a rank-local comparison): ranks that disagreed
        # about the path would wait for each other in different collectives
        flag = torch.tensor([1.0 if bad else 0.0], device=f"cuda:{local}")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        bad = bool(flag.item() > 0.5)
        if bad and (eng.use_ar_fused or eng.use_mega):
            # the fused tensor-parallel path misbehaved on this box: time the NCCL path instead (and say so).  The engine of
            # the timed run already exists: switch ITS paths off (the environment only matters at construction).
            os.environ["B200_TP_LL"] = "0"
            os.environ["B200_MEGA"] = "0"
            eng.use_ar_fused = False
            eng.use_mega = False
            eng._graphs.clear()
            tp_parity["fallback"] = "fused path rejected by the parity check; timed run uses separate kernels + NCCL all-reduce"
    _log("engine ready")
    # ---- (1) device-resident greedy loop: value ------------------------------------------------
    graph, launches_per_step = eng.capture_greedy_loop(BSZ)
    eng.tokens[:BSZ].fill_(1234)
    eng.pos[:BSZ].fill_(CTX)
    _log("graph captured")
    for _ in range(W):
        graph.replay()
    barrier()
    if world > 1 and eng.ar_fused_supported(BSZ):
        # The warm-up ran the fused tensor-parallel exchange on the FULL-SIZE model: every rank must have decoded the same
        # tokens (identical logits on all ranks is the reference's determinism contract) and no poll may have timed out.
        # Otherwise the timed run uses the NCCL all-reduce (decision all-reduced: the same on every rank).
        err = int(eng._ar["step"][1].item()) if eng._ar is not None else 0
        same, timeouts = tp_warmup_verdict(eng.tokens[:BSZ], err)
        tp_parity["full_size_warmup"] = {"ranks_decoded_same_tokens": same, "poll_timeouts": timeouts}
        if timeouts or not same:
            eng.use_ar_fused = False
            eng._graphs.clear()
            del graph
            graph, launches_per_step = eng.capture_greedy_loop(BSZ)
            eng.tokens[:BSZ].fill_(1234)
            eng.pos[:BSZ].fill_(CTX)
            for _ in range(W):
                graph.replay()
            barrier()
            tp_parity["fallback"] = ("fused exchange rejected after the full-size warm-up; timed run uses separate kernels + "
                                     "NCCL all-reduce")
    _log("warm-up done")
    clocks = ClockSampler(local) if (rank == 0 and not os.environ.get("B200_NO_CLOCKS")) else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev[0].record()
    for i in range(K):
        graph.replay()
        ev[i + 1].record()
        if os.environ.get("B200_BENCH_VERBOSE") == "2":
            torch.cuda.synchronize()
            _log(f"step {i} ok")
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.greedy_logits[:BSZ], eng.tokens[:BSZ])
    total_ms = ev[0].elapsed_time(ev[K])
    per_step = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(K))
    clk = clocks.stop() if clocks else None
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = BSZ * K / (total_ms / 1000.0)
    p50 = per_step[K // 2]

    if world > 1 and tp_parity is not None and eng.ar_fused_supported(BSZ) and eng._ar is not None:
        bad = torch.tensor([float(eng._ar["step"][1].item())], device=dev, dtype=torch.float64)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        tp_parity["poll_timeouts_timed_run"] = int(bad.item())  # non-zero: the value above was measured on a broken exchange
    _log(f"value done: {value:.1f} tok/s")
    # ---- (2) end-to-end through the public drop-in API with host buffers -------------------------
    model = B200Transformer.from_engine(eng)
    tok_host = torch.full((BSZ, 1), 1234, dtype=torch.int64).pin_memory()
    out_host = torch.zeros((BSZ,), dtype=torch.int64).pin_memory()
    tok_dev = torch.zeros((BSZ, 1), dtype=torch.int64, device=dev)

    def e2e_step(p):
        tok_dev.copy_(tok_host, non_blocking=True)                 # H2D of this step's input
        logits = model.forward_inference(tok_dev, p)               # public API (graph replay inside)
        out_host.copy_(logits.argmax(dim=-1), non_blocking=False)  # D2H of the step's result (syncs)
        tok_host[:, 0] = out_host
    pos0 = CTX + W + K + 8
    for i in range(W):
        e2e_step(pos0 + i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        e2e_step(pos0 + W + i)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = BSZ * K / (float(t.item()) / 1000.0)

    _log(f"e2e done: {e2e_value:.1f} tok/s")
    # ---- (3) roofline of the dominant kernel, measured live with CUDA events on the launching stream ----
    peak, peak_src = peaks()
    sb = eng.step_bytes(BSZ, CTX + W + K // 2)
    step_frac = (sb["total"] / (p50 / 1000.0) / 1e9) / peak
    eng.pos[:BSZ].fill_(CTX)
    if eng.mega_supported(BSZ):
        # the whole step is ONE launch of decode_step1_kernel: algorithmic bytes per launch = every packed weight,
        # the fp16 lm_head and the K/V rows [0, ctx) of all layers (SURVEY.md 8d)
        kernel_name = "b200::decode_step1_kernel (persistent whole-step kernel: 32 x [qkv, attention, wo, gate/up, down] + lm_head)"
        n_launch = 1
        bytes_per_launch = eng.step_bytes(BSZ, CTX)["total"]

        def dominant():
            eng._step(BSZ, 1, eng.cache_seq)
    else:
        kernel_name = f"b200::gemv{'1' if BSZ == 1 and cfg.bits == 4 and not cfg.group_size else ''}_kernel (qkv, wo, gate/up, down of all layers)"
        lin_bytes = 0
        n_launch = 0
        for lw in eng.layers:
            for pl in (lw.wqkv, lw.wo, lw.w13, lw.w2):
                lin_bytes += pl.nbytes
                n_launch += 1
        bytes_per_launch = lin_bytes / n_launch

        def dominant():
            # the four weight-streaming launches of every layer, same arguments as in the step (no attention)
            for i, lw in enumerate(eng.layers):
                kc, vt = eng.kcache[i], eng.vtcache[i]
                ops.gemv(lw.wqkv, BSZ, resid=eng.h[0], gamma=lw.attn_norm, eps=cfg.norm_eps, epilogue=ops.B200_EPI_QKV,
                         out=eng.q, use_pdl=eng.use_pdl,
                         qkv=dict(n_q_rows=eng.Hq * 128, n_kv_rows=eng.Hkv * 128, rope=eng.rope, pos=eng.pos,
                                  tokens_per_seq=1, kcache=kc, vtcache=vt, cache_seq=eng.cache_seq))
                ops.gemv(lw.wo, BSZ, xin=eng.attn, epilogue=ops.B200_EPI_F16, out=eng.o, use_pdl=eng.use_pdl)
                ops.gemv(lw.w13, BSZ, resid=eng.h[0], delta=eng.o, h_out=eng.h[1], gamma=lw.ffn_norm, eps=cfg.norm_eps,
                         epilogue=ops.B200_EPI_SILU, out=eng.act, use_pdl=eng.use_pdl)
                ops.gemv(lw.w2, BSZ, xin=eng.act, epilogue=ops.B200_EPI_F16, out=eng.f, use_pdl=eng.use_pdl)
    g2 = torch.cuda.CUDAGraph()
    dominant()
    torch.cuda.synchronize()
    with torch.cuda.graph(g2):
        dominant()
    for _ in range(3):
        g2.replay()
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    r0.record()
    for _ in range(reps):
        g2.replay()
    r1.record()
    torch.cuda.synchronize()
    dom_ms = r0.elapsed_time(r1) / reps
    achieved = bytes_per_launch * n_launch / (dom_ms / 1000.0) / 1e9

    # ---- (4) prompt path: one 2048-token prompt through the tensor-core prefill (weights streamed 8x instead of 64x) ----
    prefill_ms = None
    if world == 1 and eng.prefill_tc_supported():
        ptoks = torch.randint(1, MODEL["vocab_size"], (1, 2048), device=dev)
        eng.forward_inference(ptoks[:, :256], 0)  # warm-up (buffers, func attributes)
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        eng.forward_inference(ptoks, 0)
        p1.record()
        torch.cuda.synchronize()
        prefill_ms = p0.elapsed_time(p1)

    if rank != 0:
        _finish(world)
        return

    out = {
        "metric": METRIC, "value": value, "unit": "tokens/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "bits": args.bits, "group_size": args.group_size, "bsz": BSZ, "ctx": CTX,
                   "parallelism": f"tp{world}", "p50_ms_per_token": p50, "p90_ms_per_token": per_step[int(K * 0.9)],
                   "tokens_per_s_per_gpu": value / world, "l2": "inputs_exceed_l2 (3.5 GB of weights per step >> 126 MB)",
                   "pdl": eng.use_pdl, "cuda_graph": True, "step_bytes": sb,
                   "step_hbm_frac_of_peak": step_frac, "step_hbm_frac_of_8TBps": sb["total"] / (p50 / 1000.0) / 8e12,
                   "prefill_2048_ms": prefill_ms,
                   "prefill_path": "tcgen05 W4A16 GEMM (b200_prefill_gemm_w4) in 256-token chunks + decode-attention per 32 queries"},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": 8 * BSZ, "d2h_bytes_per_step": 8 * BSZ},
        "gpu_launches": launches_per_step * K,
        "roofline": {"bound": "hbm", "kernel": kernel_name,
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "frac_of_8TBps": achieved / 8000.0,
                     "peak_source": peak_src, "bytes_per_launch_avg": bytes_per_launch,
                     "launch_ms_avg": dom_ms / n_launch,
                     "traffic": ncu_traffic(kernel_name)},
    }
    if tp_parity is not None:
        out["tp_parity"] = tp_parity
    out["config"]["decode_path"] = ("persistent dataflow kernel (b200_decode_step1_ll)" if (eng.mega_supported(BSZ) and eng.mega_dataflow)
                                    else "persistent barrier kernel (b200_decode_step1)" if eng.mega_supported(BSZ)
                                    else "separate kernels (5 per layer)" + (
                                        ", all-reduce fused into the GEMVs (LL)" if eng.ar_fused_supported(BSZ) else
                                        " + NCCL all-reduce" if world > 1 else ""))
    if not args.no_cpu and world == 1:
        del graph, g2, model
        eng.destroy_kv_cache()
        v, det = cpu_decode_sample()
        out["cpu_baseline"] = {"value": v, "unit": "tokens/s", **det}
    print(json.dumps(out), flush=True)
    _finish(world)


if __name__ == "__main__":
    main()
