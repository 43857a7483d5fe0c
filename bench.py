#!/usr/bin/env python
"""bench.py -- tokens/s (bs=1) and accepted length tau of the EAGLE draft->verify->accept path.

Workload (BASELINE.json metric): Llama-3-8B-Instruct shapes + EAGLE-3 head (draft vocab 32000), bf16, batch 1,
512-token synthetic prompt, 256 new tokens, greedy, dynamic draft tree (total_token=60, top_k=10, depth=6),
random-init weights of the named shapes (no network for checkpoints).  One "step" = one
`EaModel.eagenerate(prompt, max_new_tokens=256)` call (prefill + decode cycles), as the reference times it
(eagle/evaluation/gen_ea_answer_llama3chat.py:159-169).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA engine
    python bench.py --impl reference [...]                       # the reference algorithm (CPU oracle port) on host cores
    python bench.py --dump-outputs DIR [...]                     # also write the last timed step's outputs to DIR/*.npy

Prints ONE JSON line (rank 0).  `value` is measured with the prompt already resident in HBM; `e2e` goes through
the public `EaModel.eagenerate` with a pinned-host prompt and host result (H2D/D2H inside the timed region).
`roofline` is for the dominant kernel (the tcgen05/TMA skinny weight-streaming GEMM): algorithmic weight bytes of
its launches / their CUDA-event durations, measured in extra profiled steps right after the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

import torch  # noqa: E402

PROMPT_LEN, NEW_TOKENS = 512, 256
TREE = dict(total_token=60, depth=6, top_k=10)
# --model: the targets BASELINE.json names.  eagle3 -> EAGLE-3 head (draft vocabulary 32000 + d2t), else the EAGLE-1/2 head.
MODELS = {
    "llama3-8b": dict(eagle3=True, dtype="bf16", label="llama3-8b+eagle3",
                      baseline={"dynamic": "configs[2]: Llama-3-8B-Instruct + dynamic tree (depth=6, top-k=10), bf16, bs=1 -- the tree the reference's "
                                           "eagenerate runs for the EAGLE-3 head; configs[1] (static tree) is `--tree static`",
                                "static": "configs[1]: Llama-3-8B-Instruct + EAGLE-3 head, bf16, bs=1, static draft tree"}),
    "llama2-13b": dict(eagle3=False, dtype="fp16", label="llama2-13b+eagle1",
                       baseline={"dynamic": "configs[3]: Llama-2-13B-chat + EAGLE-1 head, fp16, temperature=1.0 posterior sampling, bs=1, TP=2 "
                                            "(run with --dtype fp16 --temperature 1.0 --gpus 2)"}),
    "llama3-70b": dict(eagle3=True, dtype="bf16", label="llama3-70b+eagle3",
                       baseline={"dynamic": "configs[4]: Llama-3-70B-Instruct + EAGLE-3 head, bf16, bs=1, TP=8 (run with --gpus 8)"}),
    "vicuna-7b": dict(eagle3=False, dtype="fp16", label="vicuna-7b+eagle1",
                      baseline={"dynamic": "configs[0]: Vicuna-7B + EAGLE-1 head, greedy, bs=1 (the reference's CPU-runnable plumbing case, here on the GPU)"}),
}
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}


def tree_kwargs(tree: str) -> dict:
    if tree == "static":
        from eagle_b200.static_trees import mc_sim_7b_63
        return dict(top_k=10, tree_choices=mc_sim_7b_63)
    return dict(TREE)


def workload_name(args) -> str:
    tree = ("static-tree(mc_sim_7b_63: 26 nodes, depth 5, top_k=10)" if args.tree == "static"
            else "dynamic-tree(total_token=60,top_k=10,depth=6)")
    mode = "greedy" if args.temperature <= 1e-5 else f"sampling(T={args.temperature:g})"
    init = "random-init" if args.fixture == "random" else "correlated-init(permutation-bigram target + copy head, 25% of draft rows corrupted)"
    layers = "" if not args.layers else f" layers={args.layers}"
    return f"{MODELS[args.model]['label']} {args.dtype} bs1 {PROMPT_LEN}in/{NEW_TOKENS}out {mode} {tree} {init}{layers}"


def baseline_config(args) -> str:
    """Which BASELINE.json `configs` entry the run corresponds to."""
    b = MODELS[args.model]["baseline"]
    return b.get(args.tree, b["dynamic"])


def profile_traffic_ratio():
    """DRAM bytes / algorithmic bytes of the dominant kernel, measured with `ncu --set full` by tools/final_run.sh and stored in
    profiles/ (dram__bytes_read.sum + dram__bytes_write.sum per launch over the weight bytes of that launch)."""
    p = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["dram_over_algorithmic"]), d.get("source", p)
    return None, "no ncu traffic capture committed for this kernel yet"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# model shapes and synthetic weights (shared by both arms)
# ------------------------------------------------------------------------------------------------------
def model_configs(args):
    from eagle_b200 import synthetic as syn
    spec = MODELS[args.model]
    tcfg = syn.target_config(args.model)
    if args.layers:
        tcfg["num_hidden_layers"] = args.layers
    if spec["eagle3"]:
        hcfg = syn.head_config(args.model, True, draft_vocab_size=32000)
    else:
        hcfg = syn.head_config(args.model, False)
    return tcfg, hcfg, spec["eagle3"]


def weight_specs(tcfg, hcfg, eagle3):
    """(which, name, shape, kind) for every tensor of the target ("t") and the head ("h"); kind: normal | ones | zeros."""
    H, I, V, L = tcfg["hidden_size"], tcfg["intermediate_size"], tcfg["vocab_size"], tcfg["num_hidden_layers"]
    A, kvd = tcfg["num_attention_heads"] * 128, tcfg["num_key_value_heads"] * 128
    yield "t", "model.embed_tokens.weight", (V, H), "normal"
    for i in range(L):
        p = f"model.layers.{i}."
        yield "t", p + "self_attn.q_proj.weight", (A, H), "normal"
        yield "t", p + "self_attn.k_proj.weight", (kvd, H), "normal"
        yield "t", p + "self_attn.v_proj.weight", (kvd, H), "normal"
        yield "t", p + "self_attn.o_proj.weight", (H, A), "normal"
        yield "t", p + "mlp.gate_proj.weight", (I, H), "normal"
        yield "t", p + "mlp.up_proj.weight", (I, H), "normal"
        yield "t", p + "mlp.down_proj.weight", (H, I), "normal"
        yield "t", p + "input_layernorm.weight", (H,), "ones"
        yield "t", p + "post_attention_layernorm.weight", (H,), "ones"
    yield "t", "model.norm.weight", (H,), "ones"
    yield "t", "lm_head.weight", (V, H), "normal"
    Hh, Ih = hcfg["hidden_size"], hcfg["intermediate_size"]
    hA, hkvd = hcfg["num_attention_heads"] * 128, hcfg["num_key_value_heads"] * 128
    if eagle3:
        pre, qk_in = "midlayer.", 2 * Hh
        yield "h", "fc.weight", (Hh, 3 * H), "normal"
        yield "h", "norm.weight", (Hh,), "ones"
        yield "h", "lm_head.weight", (hcfg["draft_vocab_size"], Hh), "normal"
        yield "h", pre + "hidden_norm.weight", (Hh,), "ones"
        yield "h", pre + "input_layernorm.weight", (Hh,), "ones"
    else:
        pre, qk_in = "layers.0.", Hh
        yield "h", "fc.weight", (Hh, 2 * Hh), "normal"
        yield "h", "fc.bias", (Hh,), "zeros"
    yield "h", pre + "post_attention_layernorm.weight", (Hh,), "ones"
    yield "h", pre + "self_attn.q_proj.weight", (hA, qk_in), "normal"
    yield "h", pre + "self_attn.k_proj.weight", (hkvd, qk_in), "normal"
    yield "h", pre + "self_attn.v_proj.weight", (hkvd, qk_in), "normal"
    yield "h", pre + "self_attn.o_proj.weight", (Hh, hA), "normal"
    yield "h", pre + "mlp.gate_proj.weight", (Ih, Hh), "normal"
    yield "h", pre + "mlp.up_proj.weight", (Ih, Hh), "normal"
    yield "h", pre + "mlp.down_proj.weight", (Hh, Ih), "normal"


def weight_bytes_per_cycle(tcfg, hcfg, eagle3, depth):
    """SURVEY 8(d): algorithmic bytes of one draft->verify->accept cycle = every target matrix once (verify) + the head's
    matrices once per draft pass (1 stable + depth tree levels; the EAGLE-3 fc only in the stable pass)."""
    t = h = fc = 0
    for which, name, shape, kind in weight_specs(tcfg, hcfg, eagle3):
        if kind != "normal" or "embed" in name:
            continue
        n = 2 * shape[0] * shape[1]
        if which == "t":
            t += n
        elif name == "fc.weight" and eagle3:
            fc += n
        else:
            h += n
    if not eagle3:
        h += 2 * tcfg["vocab_size"] * tcfg["hidden_size"]  # the EAGLE-1 head scores with the target's lm_head
    return t + fc + (1 + depth) * h, t


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the CPU oracle port of the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------------
def _tiled_normal(shape, base, offset, dtype):
    """Random-init weights for the CPU arm without paying 5 minutes of host RNG for 8e9 elements: every tensor is
    filled from one 64 Mi-element N(0, 0.02) block read at a per-tensor offset (distinct memory, same statistics)."""
    n = 1
    for s in shape:
        n *= s
    out = torch.empty(n, dtype=dtype)
    pos, blen = 0, base.numel()
    off = offset % blen
    while pos < n:
        take = min(n - pos, blen - off)
        out[pos:pos + take] = base[off:off + take]
        pos += take
        off = 0
    return out.view(*shape)


def effective_cores() -> int:
    """Cores this process may actually use: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def numa_node0_cpus():
    """CPUs of NUMA node 0 that this process may use (the 96-thread 8-GPU hosts are two sockets: a weight-streaming CPU run that
    spans both is several times slower than one pinned to a socket -- VERDICT r1 weak #9)."""
    try:
        with open("/sys/devices/system/node/node0/cpulist") as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        return sorted(cpus & allowed)
    except Exception:
        return []


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def cpu_reference_run(args, cycles: int, threads: int):
    """Prefill 512 tokens + `cycles` draft->verify->accept cycles of the oracle port (oracle/eagle_oracle.py, a restatement
    of the reference's eagenerate).  Returns (extrapolated tokens/s for the 256-token job, tau, detail dict).  The thread count
    is SWEPT on single verify-sized forwards first and the fastest setting is used: the baseline is the best CPU number."""
    from oracle import eagle_oracle as orc
    from eagle_b200 import synthetic as syn
    dtype = DTYPES[args.dtype]
    tcfg, hcfg, eagle3 = model_configs(args)
    node0 = numa_node0_cpus()
    if node0 and len(node0) < len(os.sched_getaffinity(0)):
        os.sched_setaffinity(0, node0)  # one socket: local memory for the 16 GB of weights
        threads = min(threads, len(node0))
        log(f"cpu reference arm pinned to NUMA node 0 ({len(node0)} cpus)")
    torch.set_num_threads(threads)
    log(f"cpu reference arm: up to {threads} threads, building {MODELS[args.model]['label']} shaped weights on the host")
    g = torch.Generator().manual_seed(0)
    base = torch.empty(1 << 26, dtype=dtype).normal_(0, 0.02, generator=g)
    t0 = time.time()
    tW, hW, cnt = {}, {}, 0
    for which, name, shape, kind in weight_specs(tcfg, hcfg, eagle3):
        cnt += 1
        if kind == "normal":
            w = _tiled_normal(shape, base, cnt * 7919 * 4099, dtype)
        else:
            w = torch.ones(shape, dtype=dtype) if kind == "ones" else torch.zeros(shape, dtype=dtype)
        (tW if which == "t" else hW)[name] = w
    hW["embed_tokens.weight"] = tW["model.embed_tokens.weight"]
    if eagle3:
        hW["d2t"], hW["t2d"] = syn.make_d2t(tcfg["vocab_size"], hcfg["draft_vocab_size"])
    build_s = time.time() - t0
    keys = orc.ModelCfg.__dataclass_fields__.keys()
    m = orc.OracleEaModel(orc.ModelCfg(**{k: v for k, v in tcfg.items() if k in keys}), tW,
                          orc.ModelCfg(**{k: v for k, v in hcfg.items() if k in keys}), hW, eagle3, **tree_kwargs(args.tree))
    V = tcfg["vocab_size"]
    prompt = torch.randint(0, V - 200, (1, PROMPT_LEN), generator=torch.Generator().manual_seed(0))
    # untimed warm-up (first touch of the weights), thread sweep on one 60-row target forward, then the timed run
    log(f"weights built in {build_s:.1f} s; warm-up pass (prefill + 1 cycle)")
    t = time.time()
    m.eagenerate(prompt, max_new_tokens=0, max_length=2048, log=True)
    log(f"warm-up took {time.time() - t:.1f} s")
    sweep = {}
    cands = sorted({c for c in (8, 16, 24, 32, 48, threads) if c <= threads})
    probe = torch.randint(0, V - 200, (1, 60), generator=torch.Generator().manual_seed(1))
    for c in cands:
        torch.set_num_threads(c)
        kv = m._kv(2048)
        m.target.forward(probe, kv)
        t = time.time()
        m.target.forward(probe, m._kv(2048))
        sweep[c] = round(time.time() - t, 3)
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    log(f"thread sweep (s per 60-row target forward): {sweep} -> {best} threads; timed pass with {cycles} cycles")
    m.time_log = []
    ids, new_token, idx = m.eagenerate(prompt, max_new_tokens=max(0, cycles - 1), max_length=2048, log=True)
    tl = m.time_log
    n_cyc = idx + 1
    prefill_s = tl[1] - tl[0]
    cyc_s = (tl[-1] - tl[1]) / n_cyc
    tau = new_token / n_cyc
    job_cycles = (NEW_TOKENS + 1) / tau  # eagenerate stops once new_token > max_new_tokens
    job_s = prefill_s + job_cycles * cyc_s
    toks = (job_cycles * tau) / job_s
    detail = dict(prefill_s=round(prefill_s, 2), cycle_s=round(cyc_s, 3), cycles_timed=n_cyc, tau=round(tau, 3),
                  weight_build_s=round(build_s, 1), thread_sweep_s=sweep, threads=best, numa_pinned=bool(node0))
    return toks, tau, detail


def torch_cuda_reference_run(args, cycles: int):
    """BASELINE.md 2's "practical bar": the reference ALGORITHM as eager PyTorch ops on the B200 itself (the oracle port with its
    tensors on `cuda`; the reference proper cannot travel to the GPU box).  Same extrapolation as the CPU arm."""
    from oracle import eagle_oracle as orc
    from eagle_b200 import synthetic as syn
    dtype = DTYPES[args.dtype]
    tcfg, hcfg, eagle3 = model_configs(args)
    V = tcfg["vocab_size"]
    prompt = torch.randint(0, V - 200, (1, PROMPT_LEN), generator=torch.Generator().manual_seed(0)).cuda()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    tW, hW = {}, {}
    for which, name, shape, kind in weight_specs(tcfg, hcfg, eagle3):
        if kind == "normal":
            w = (torch.randn(shape, generator=gen, device="cuda", dtype=torch.float32) * 0.02).to(dtype)
        else:
            w = torch.ones(shape, dtype=dtype, device="cuda") if kind == "ones" else torch.zeros(shape, dtype=dtype, device="cuda")
        (tW if which == "t" else hW)[name] = w
    hW["embed_tokens.weight"] = tW["model.embed_tokens.weight"]
    if eagle3:
        d2t, t2d = syn.make_d2t(V, hcfg["draft_vocab_size"])
        hW["d2t"], hW["t2d"] = d2t.cuda(), t2d.cuda()
    torch.set_default_device("cuda")  # every tensor the port creates (masks, position ids, KV) now lives on the GPU
    keys = orc.ModelCfg.__dataclass_fields__.keys()
    m = orc.OracleEaModel(orc.ModelCfg(**{k: v for k, v in tcfg.items() if k in keys}), tW,
                          orc.ModelCfg(**{k: v for k, v in hcfg.items() if k in keys}), hW, eagle3, **tree_kwargs(args.tree))
    m.eagenerate(prompt, max_new_tokens=0, max_length=2048, log=True)  # warm-up
    torch.cuda.synchronize()
    m.time_log = []
    _orig_time = time.time

    def synced_time():
        torch.cuda.synchronize()
        return _orig_time()

    orc.time.time = synced_time  # the port stamps wall-clock time after prefill and after every cycle
    try:
        ids, new_token, idx = m.eagenerate(prompt, max_new_tokens=max(0, cycles - 1), max_length=2048, log=True)
    finally:
        orc.time.time = _orig_time
    tl = m.time_log
    n_cyc = idx + 1
    prefill_s = tl[1] - tl[0]
    cyc_s = (tl[-1] - tl[1]) / n_cyc
    tau = new_token / n_cyc
    job_cycles = (NEW_TOKENS + 1) / tau
    toks = (job_cycles * tau) / (prefill_s + job_cycles * cyc_s)
    return toks, tau, dict(prefill_s=round(prefill_s, 4), cycle_s=round(cyc_s, 4), cycles_timed=n_cyc)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.ref_device == "cuda":
        toks, tau, detail = torch_cuda_reference_run(args, cycles=max(4, min(24, args.steps + args.warmup)))
        print(json.dumps({"impl": "reference-eager-torch-on-cuda", "metric": "tokens/sec (bs=1)", "value": round(toks, 3), "unit": "tokens/s",
                          "tau": round(tau, 3), "dtype": args.dtype, "config": {"workload": workload_name(args)}, "detail": detail,
                          "what": "the CPU oracle port (reference algorithm, eager torch ops, HF-style dense masks, Python tree bookkeeping) with its "
                                  "tensors on the B200; extrapolated to the 256-token job from measured prefill and per-cycle times"}), flush=True)
        return
    cores = min(effective_cores(), args.cpu_threads) if args.cpu_threads > 0 else effective_cores()
    cycles = max(2, args.steps + args.warmup)
    toks, tau, detail = cpu_reference_run(args, cycles=min(cycles, 12), threads=cores)
    sample = (f"{PROMPT_LEN}-token prefill + {detail['cycles_timed']} draft->verify->accept cycles of the full {MODELS[args.model]['label']} shapes; "
              f"tokens/s extrapolated to the {NEW_TOKENS}-token job from measured prefill {detail['prefill_s']} s and {detail['cycle_s']} s/cycle; "
              f"best of a thread sweep {detail['thread_sweep_s']} (one NUMA node when the host has several); "
              "weights tiled from a 64Mi-element N(0,0.02) block")
    line = {"impl": "reference", "metric": "tokens/sec (bs=1)", "value": round(toks, 4), "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1000.0 * (NEW_TOKENS + 1) / toks, 1),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "tau": round(tau, 3),
            "config": {"workload": workload_name(args), "baseline": baseline_config(args), "parallelism": f"tp{args.gpus}", "l2": "inputs larger than L2"},
            "cpu_baseline": {"value": round(toks, 4), "unit": "tokens/s", "cores": detail["threads"], "kind": "port", "sample": sample},
            "e2e": {"value": round(toks, 4), "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "detail": detail}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def build_engine(args, device: int, tp_rank: int, tp_size: int):
    from eagle_b200 import EaModel, synthetic as syn
    dtype = DTYPES[args.dtype]
    tcfg, hcfg, eagle3 = model_configs(args)
    dev = f"cuda:{device}"
    if args.fixture == "correlated":
        if args.model != "llama3-8b":
            raise SystemExit("--fixture correlated is defined for --model llama3-8b")
        m = EaModel(tcfg, syn.head_config(args.model, True, draft_vocab_size=32000, num_key_value_heads=tcfg["num_attention_heads"]),
                    use_eagle3=True, torch_dtype=dtype, device=device, max_length=2048, tp_rank=tp_rank, tp_size=tp_size, **tree_kwargs(args.tree))
        if tp_size > 1:
            m.init_tp()
        _, tW, _, hW = syn.correlated_llama3_eagle3(tcfg["num_hidden_layers"], dtype, dev)
        m.load_target_state_dict(tW)
        m.load_head_state_dict(hW)
        del tW, hW
        torch.cuda.empty_cache()
        m.finalize()
        return m, tcfg, hcfg, eagle3
    m = EaModel(tcfg, hcfg, use_eagle3=eagle3, torch_dtype=dtype, device=device, max_length=2048, tp_rank=tp_rank, tp_size=tp_size,
                **tree_kwargs(args.tree))
    if tp_size > 1:
        m.init_tp()  # every rank generates the same full tensors (same seed); the engine keeps only its shard
    # stream the random-init weights tensor by tensor (never more than one extra tensor resident)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    for which, name, shape, kind in weight_specs(tcfg, hcfg, eagle3):
        if kind == "normal":
            w = (torch.randn(shape, generator=gen, device=dev, dtype=torch.float32) * 0.02).to(dtype)
        else:
            w = torch.ones(shape, dtype=dtype, device=dev) if kind == "ones" else torch.zeros(shape, dtype=dtype, device=dev)
        m._load(name if which == "t" else "head." + name, w)
        del w
    if eagle3:
        d2t, _ = syn.make_d2t(tcfg["vocab_size"], hcfg["draft_vocab_size"])
        m._load("head.d2t", d2t)
    m.finalize()
    return m, tcfg, hcfg, eagle3


def tp_parity_check(world: int, rank: int, device: int):
    """Tensor-parallel token parity INSIDE the bench run (VERDICT r1 next #1a): the reference-generated goldens
    (tests/golden/*.pt, produced by the unmodified reference, oracle/make_golden.py) are replayed through an engine sharded over
    all `world` ranks before the timed region; any mismatch fails the run."""
    from eagle_b200 import EaModel, synthetic as syn
    fixtures = ["e3_tp8_bf16"] + (["e3_gqa_bf16", "e1_corr_fp16"] if world == 2 else [])
    out = []
    for fx in fixtures:
        g = torch.load(os.path.join(ROOT, "tests", "golden", fx + ".pt"), weights_only=False)
        tcfg, tW, hcfg, hW, eagle3, dtype, tree = syn.fixture_models(fx)
        m = EaModel.from_state_dicts(tcfg, tW, hcfg, hW, use_eagle3=eagle3, torch_dtype=dtype, max_length=512, device=device,
                                     tp_rank=rank, tp_size=world, **tree)
        ids, new_token, idx = m.eagenerate(g["prompt"].cuda(), log=True, **g["gen_kw"])
        ok = ids.cpu().tolist() == g["ids"].tolist()
        out.append({"fixture": fx, "ids_match": bool(ok), "new_token": [int(new_token), int(g["new_token"])], "idx": [int(idx), int(g["idx"])]})
        torch.cuda.synchronize()
        torch.distributed.barrier()  # no rank frees its peer window while another rank may still be inside its last cycle
        del m
    return out


def timed_steps(m, prompt, steps, dist, gen_kw):
    """K eagenerate calls bracketed by barrier + synchronize, timed with CUDA events on the engine's stream.  Also returns what
    the last call returned: (ids, new_token, idx)."""
    stream = m.cuda_stream()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    new_tokens, cycles, last = 0, 0, None
    for _ in range(steps):
        last = m.eagenerate(prompt, max_new_tokens=NEW_TOKENS, max_length=2048, log=True, **gen_kw)
        new_tokens += last[1]
        cycles += last[2] + 1
    e1.record(stream)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1), new_tokens, cycles, last


def dump_outputs(directory, ids, new_token, idx):
    """Write what one `eagenerate(..., log=True)` call returns as float64 .npy files (token ids are exact in float64), so that
    two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, value in (("ids", ids.cpu().numpy()), ("new_token", new_token), ("idx", idx)):
        np.save(os.path.join(directory, name + ".npy"), np.asarray(value, dtype=np.float64))


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- eagle_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        dist = dist_mod
    tp_parity = None
    if world > 1:
        log(f"tp{world} token parity on the reference goldens")
        tp_parity = tp_parity_check(world, rank, local)
        flags = torch.tensor([int(all(p["ids_match"] and p["new_token"][0] == p["new_token"][1] and p["idx"][0] == p["idx"][1] for p in tp_parity))],
                             device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if int(flags[0]) != 1:
            raise SystemExit(f"bench.py: tensor-parallel token parity FAILED on rank {rank}: {tp_parity}")
    log(f"building the engine ({workload_name(args)}), tp{world} rank {rank}")
    m, tcfg, hcfg, eagle3 = build_engine(args, local, rank, world)
    log("engine ready; warm-up")
    V = tcfg["vocab_size"]
    if args.fixture == "correlated":
        from eagle_b200 import synthetic as syn
        used = syn.draft_vocab_ids(V, 32000)
        prompt_host = used[torch.randint(0, used.numel(), (PROMPT_LEN,), generator=torch.Generator().manual_seed(0))][None].pin_memory()
    else:
        prompt_host = torch.randint(0, V - 200, (1, PROMPT_LEN), generator=torch.Generator().manual_seed(0)).pin_memory()
    prompt_dev = prompt_host.cuda()
    gen_kw = dict(temperature=args.temperature) if args.temperature > 1e-5 else {}
    torch.manual_seed(1234)
    for _ in range(max(3, args.warmup)):
        m.eagenerate(prompt_dev, max_new_tokens=NEW_TOKENS, max_length=2048, **gen_kw)
    m.reset_stats()
    sampler = ClockSampler(local)
    sampler.start()
    log("timed region")
    ms_dev, new_tokens, cycles, last = timed_steps(m, prompt_dev, args.steps, dist, gen_kw)   # inputs resident in HBM
    st = m.stats()
    launches = st["kernel_launches"]
    chain_stats = {k: st[k] for k in ("chain_ms", "chain_bytes", "chain_launches")}
    ms_e2e, new_tokens_e, _, _ = timed_steps(m, prompt_host, args.steps, dist, gen_kw)     # pinned-host prompt, host result
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    if dist is not None:
        t = torch.tensor([ms_dev, ms_e2e], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
    value = new_tokens / (ms_dev / 1e3)
    e2e = new_tokens_e / (ms_e2e / 1e3)
    tau = new_tokens / max(1, cycles)
    log(f"timed: {value:.1f} tok/s device-resident, {e2e:.1f} tok/s end to end; profiling steps")
    # ---- prefill share, measured separately (512-token prefill + first tree)
    stream = m.cuda_stream()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    pe0.record(stream)
    for _ in range(3):
        m.prefill(prompt_dev)
    pe1.record(stream)
    torch.cuda.synchronize()
    prefill_ms = pe0.elapsed_time(pe1) / 3
    # ---- roofline of the dominant kernel.  (1) whole-cycle view from the timed region itself: algorithmic weight bytes of a cycle /
    # (device time of the decode cycles) -- no profiler, no eager mode, graph replay as timed; (2) per-launch view: CUDA events
    # around every launch in extra eager steps (upper bound on the in-graph kernel time).
    peak, peak_src = measured_peaks()
    cyc_bytes, verify_bytes = weight_bytes_per_cycle(tcfg, hcfg, eagle3, TREE["depth"] if args.tree != "static" else 5)
    decode_ms = ms_dev / args.steps - prefill_ms
    cycles_per_step = cycles / args.steps
    cycle_ms = decode_ms / max(1.0, cycles_per_step)
    # under TP every rank streams its shard of the target and the whole (replicated) head
    per_rank_cycle_bytes = (cyc_bytes - verify_bytes) + verify_bytes / world
    ach_cycle = per_rank_cycle_bytes / 1e9 / (cycle_ms / 1e3) if cycle_ms > 0 else 0.0
    m.reset_stats()
    m.set_profiling(True)
    for _ in range(max(1, min(2, args.steps))):
        m.eagenerate(prompt_dev, max_new_tokens=NEW_TOKENS, max_length=2048, **gen_kw)
    ps = m.stats()
    m.set_profiling(False)
    ach = ps["gemm_bytes"] / 1e9 / (ps["gemm_ms"] / 1e3) if ps["gemm_ms"] > 0 else 0.0
    vach = ps["verify_gemm_bytes"] / 1e9 / (ps["verify_gemm_ms"] / 1e3) if ps["verify_gemm_ms"] > 0 else 0.0
    total_ms = ps["gemm_ms"] + ps["attn_ms"] + ps["other_ms"]
    ratio, ratio_src = profile_traffic_ratio()
    chain = bool(os.environ.get("EB200_CHAIN", "") == "1")
    roofline = {"kernel": ("gemm_chain_kernel (persistent per-layer chain: TMA + tcgen05.mma weight streaming, stream-K, fused RMSNorm / SwiGLU / RoPE / "
                           "arg-max finishes) + skinny_gemm_tcgen05 (draft head), all launches") if chain else
                          "skinny_gemm_tcgen05 (TMA + tcgen05.mma weight-streaming GEMM, cluster split-K; lm_head as a reduction-free chain launch "
                          "with fused arg-max), all launches",
                "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": round(ratio * ps["gemm_bytes"] / max(1, ps["gemm_launches"])) if ratio else None,
                "traffic_source": ratio_src, "peak_source": peak_src, "launches": int(ps["gemm_launches"]),
                "bytes_per_launch_avg": round(ps["gemm_bytes"] / max(1, ps["gemm_launches"])),
                "us_per_launch_avg": round(1e3 * ps["gemm_ms"] / max(1, ps["gemm_launches"]), 2),
                "verify_gemm": {"achieved": round(vach, 1), "frac": round(vach / peak, 4)},
                "share_of_kernel_time": {"gemm": round(ps["gemm_ms"] / total_ms, 3), "attention": round(ps["attn_ms"] / total_ms, 3),
                                         "other": round(ps["other_ms"] / total_ms, 3)} if total_ms > 0 else None,
                "how": "per-launch CUDA events on the engine stream over profiled (eager) eagenerate steps run right after the timed region: "
                       "an upper bound on the in-graph kernel time",
                "in_graph": ({"kernel": "gemm_chain_kernel", "achieved": round(chain_stats["chain_bytes"] / 1e9 / (chain_stats["chain_ms"] / 1e3), 1),
                              "frac": round(chain_stats["chain_bytes"] / 1e9 / (chain_stats["chain_ms"] / 1e3) / peak, 4),
                              "launches": int(chain_stats["chain_launches"]),
                              "us_per_launch_avg": round(1e3 * chain_stats["chain_ms"] / max(1, chain_stats["chain_launches"]), 2),
                              "bytes_per_launch_avg": round(chain_stats["chain_bytes"] / max(1, chain_stats["chain_launches"])),
                              "share_of_step": round(chain_stats["chain_ms"] / (ms_dev), 4),
                              "how": "%globaltimer stamps taken INSIDE the kernel during the timed region (graph replay, no profiler): from "
                                     "'dependencies resolved' on CTA 0 to the exit of the last CTA, summed over launches; algorithmic weight "
                                     "bytes of those launches"} if chain_stats["chain_ms"] > 0 else None),
                "whole_cycle": {"achieved": round(ach_cycle, 1), "frac": round(ach_cycle / peak, 4), "cycle_ms": round(cycle_ms, 4),
                                "bytes_per_cycle_per_rank": round(per_rank_cycle_bytes), "prefill_ms": round(prefill_ms, 3),
                                "how": "algorithmic weight bytes of one draft->verify->accept cycle (SURVEY 8d) / the device time of the decode "
                                       "cycles inside the timed region (graph replay, no profiler): every non-GEMM kernel and every gap counts "
                                       "against it"}}
    line = {"metric": "tokens/sec (bs=1)", "value": round(value, 3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": round(ms_dev / args.steps, 2), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "tau": round(tau, 3),
            "config": {"workload": workload_name(args), "baseline": baseline_config(args), "parallelism": f"tp{world}",
                       "l2": "inputs larger than L2"},
            "weights_gb_per_cycle": round(cyc_bytes / 1e9, 2),
            "clocks": clocks,
            "e2e": {"value": round(e2e, 3), "unit": "tokens/s", "ms_per_step": round(ms_e2e / args.steps, 2), "h2d_bytes_per_step": PROMPT_LEN * 8,
                    "d2h_bytes_per_step": int((PROMPT_LEN + new_tokens_e / args.steps) * 8)},
            "gpu_launches": int(launches), "launches_per_cycle": round(launches / max(1, cycles), 1), "prefill_ms": round(prefill_ms, 3),
            "roofline": roofline}
    if tp_parity is not None:
        line["tp_parity"] = tp_parity
        line["tp_data_path"] = (("two-shot (row owners)" if world >= int(os.environ.get("EB200_TP_TWO_SHOT_MIN", "8")) else "one-shot") +
                                " all-reduce + residual + RMSNorm kernel over NVLink peer windows (CUDA IPC) behind every row-parallel "
                                "projection, vocabulary-parallel arg-max exchanged through the same windows: no NCCL call on the decode path"
                                if getattr(m, "tp_fused", False) else "NCCL all-reduce per row-parallel projection")
        # bytes each rank pushes over NVLink per cycle, 2 row-parallel projections per layer.  one-shot: the fp32 row to every peer;
        # two-shot: the fp32 row to its owner ((tp-1)/tp of the rows) + the owner's bf16 x and xn rows to every peer (rows/tp each)
        rows = TREE["total_token"] if args.tree != "static" else 26
        H_, L_ = tcfg["hidden_size"], tcfg["num_hidden_layers"]
        if world >= int(os.environ.get("EB200_TP_TWO_SHOT_MIN", "8")):
            per_proj = rows * H_ * 4 * (world - 1) / world + (rows / world) * (world - 1) * H_ * 2 * 2
        else:
            per_proj = (world - 1) * rows * H_ * 4
        line["nvlink_push_bytes_per_cycle_per_rank"] = int(per_proj * 2 * L_) if getattr(m, "tp_fused", False) else None
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            # the CPU arm runs in a child process with a hard deadline so that a slow host can never stall the GPU result
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(max(1, args.cpu_cycles - 1)),
                   "--warmup", "1", "--cpu-threads", str(args.cpu_threads), "--tree", args.tree, "--model", args.model, "--dtype", args.dtype]
            if args.layers:
                cmd += ["--layers", str(args.layers)]
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=args.cpu_timeout, cwd=ROOT)
                ref = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
                line["cpu_baseline"]["tau"] = ref.get("tau")
            except subprocess.TimeoutExpired:
                line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": effective_cores(), "kind": "port",
                                        "sample": f"CPU arm exceeded its {args.cpu_timeout} s budget on this host (run `bench.py --impl reference`)"}
            except Exception as ex:
                line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": effective_cores(), "kind": "port",
                                        "sample": f"CPU arm failed: {ex!r}"}
            # BASELINE.md 2: the reference algorithm as eager PyTorch on this same B200 (extra key; own child process)
            try:
                cmd2 = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-device", "cuda", "--steps", "10", "--warmup", "2",
                        "--tree", args.tree, "--model", args.model, "--dtype", args.dtype]
                if args.layers:
                    cmd2 += ["--layers", str(args.layers)]
                out2 = subprocess.run(cmd2, capture_output=True, text=True, timeout=180, cwd=ROOT)
                ref2 = json.loads([l for l in out2.stdout.splitlines() if l.startswith("{")][-1])
                line["eager_torch_on_b200"] = {"value": ref2["value"], "unit": "tokens/s", "tau": ref2["tau"], "detail": ref2["detail"], "what": ref2["what"]}
            except Exception as ex:
                line["eager_torch_on_b200"] = {"value": None, "error": repr(ex)[:300]}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tree", default="dynamic", choices=["dynamic", "static"],
                    help="dynamic = the headline workload (EAGLE-2/3 re-ranked tree); static = the reference's fixed mc_sim_7b_63 tree")
    ap.add_argument("--model", default="llama3-8b", choices=sorted(MODELS), help="target shapes (BASELINE.json configs); default = the headline")
    ap.add_argument("--dtype", default=None, choices=sorted(DTYPES), help="model dtype (default: the one BASELINE.json names for --model)")
    ap.add_argument("--temperature", type=float, default=0.0, help="> 0: the sampling posterior (configs[3] runs at 1.0)")
    ap.add_argument("--fixture", default="random", choices=["random", "correlated"],
                    help="random = random-init weights (tau = 1, the headline); correlated = bigram target + copy head at the same shapes (tau > 1)")
    ap.add_argument("--layers", type=int, default=0, help="override the number of target layers (debugging; 0 = the model's own)")
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference only: cpu = the driver's reference arm (host cores); cuda = the same port as eager PyTorch on the GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-cycles", type=int, default=6)
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU arm (0 = all effective cores)")
    ap.add_argument("--cpu-timeout", type=int, default=240)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last device-resident timed step returned (ids, new_token, idx) to DIR/<name>.npy as float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dtype is None:
        args.dtype = MODELS[args.model]["dtype"]
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
