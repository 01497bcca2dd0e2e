#!/usr/bin/env python
"""Headline benchmark: decode tokens/s of the TriForce hierarchy at a 128K prompt (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (N = 1, BASELINE.json configs[1]): Llama2-7B-128K shapes (random-init fp16 weights — no checkpoints offline),
on-chip, prefill = 124928 synthetic tokens, retrieval budget 4096, chunk 8, gamma 6, T = 0.6, top-p 0.9.
A STEP is one outer TriForce iteration: Middle_Spec (draft ↔ retrieval-cache verify) + one (gamma2+1)-row verify over the
full KV + accept/resample + cache maintenance; it yields a data-dependent number of tokens.  `value` = tokens produced
by the K timed steps / device time (CUDA events, max over ranks).  Also reported: the autoregressive baseline measured in
the same process (one full-KV decode step per token, captured as a CUDA graph — faster than the reference's eager loop,
so the speed-up quoted is conservative), average accepted length, the KV-read roofline of the dominant kernel, and a CPU
baseline of the same path (the numpy oracle port, bounded sample).

N > 1 (torchrun): the same workload head-sharded over N GPUs (tensor parallel, NCCL all-reduce on the o_proj / down_proj
seams — the reference's own scheme, models/TP_llama.py), i.e. STRONG scaling.

Also in the `ours` line (N = 1): `acceptance_sweep` (the same job on acceptance-calibrated synthetic weights — the regime the
reference's 2.2x lives in), `reference_gpu` (the UNMODIFIED reference from baseline/_ref with real flash-attn + its CUDA graphs on
the same B200, same shapes and weights: its Autoregressive ms/token and TriForce tokens/s) and `roofline.vs_fa2` (flash-attn's
FA2 kernel through the reference's own call next to tf_verify_attn).

`--impl reference`: the reference's own Python (baseline/_ref, staged by __graft_entry__.build(); baseline/run_reference.py
documents the shims) on the host CPU cores: its HF-eager path with fp32 weights, exactly W + K outer iterations of its own
TriForce loop at the same shapes, K of them timed.  Bounded sample: the prompt KV is synthetic instead of prefilled on the CPU.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "decode tokens/sec at 128K prefill (TriForce, Llama2-7B-128K shapes, budget 4096, gamma 6)"
UNIT = "tokens/s"
# the line of the last `--impl reference` run on this host, reused as the `cpu_baseline` of a later `ours` run (outside the tree,
# which may be read-only)
REFERENCE_LAST = os.path.join(tempfile.gettempdir(), "triforce_b200_reference_last.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--target", default="llama-7B-128K")
    ap.add_argument("--prefill", type=int, default=124928)
    ap.add_argument("--budget", type=int, default=4096)
    ap.add_argument("--chunk_size", type=int, default=8)
    ap.add_argument("--gamma", type=int, default=6)
    ap.add_argument("--temp", type=float, default=0.6)
    ap.add_argument("--top_p", type=float, default=0.9)
    ap.add_argument("--gen_len", type=int, default=1024, help="KV capacity reserved for generated tokens")
    ap.add_argument("--ar_steps", type=int, default=24)
    ap.add_argument("--prefill_chunk", type=int, default=1024, help="target prefill chunk (untimed; reference uses 128)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--cpu_seconds", type=float, default=20.0)
    ap.add_argument("--attn_variant", type=int, default=0)
    ap.add_argument("--weights", default="random", help="'random' (default: plain random-init) or 'agreement:a_t,a_d' "
                    "(acceptance-calibrated synthetic weights, see triforce_b200/synth.py)")
    ap.add_argument("--sweep", default="0.003,0.001,0.0", help="acceptance sweep: agreement alphas, descending ('' = skip; N = 1 only)")
    ap.add_argument("--sweep_steps", type=int, default=16)
    ap.add_argument("--no_reference_gpu", action="store_true", help="skip the reference-on-this-GPU leg (N = 1 only)")
    ap.add_argument("--time_budget", type=float, default=690.0,
                    help="seconds the whole invocation may take: optional legs that would overrun it are skipped and say so")
    ap.add_argument("--no_traffic_probe", action="store_true", help="skip the ncu child that counts the DRAM bytes of one attention launch (N = 1 only)")
    ap.add_argument("--reference_gpu_timeout", type=int, default=600)
    ap.add_argument("--tree_size", default="512")
    ap.add_argument("--loop", default="device", choices=["device", "host"],
                    help="device (default): one CUDA-graph launch per outer step, Middle_Spec as a device-side WHILE node "
                         "(triforce_b200/device_loop.py); host: the step-wise loop (decoding.TriForceRun, one host sync per inner iteration)")
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configs[1..3]: cfg2 = 7B-128K P 124928 B 4096 gamma 6 (default); cfg3 = LWM shapes (plain RoPE), "
                         "P 130048; cfg4 = 7B-128K P 130048 B 12288 gamma 16 (the TP configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR: tokens.npy (the tokens it produced, "
                         "float64) and target_probs.npy (the target's probabilities at the rows it verified over the full KV, float32). "
                         "The full-KV attention then keeps its equal key split (TRIFORCE_ATTN_CALIBRATE=0), so the outputs are "
                         "bit-reproducible from run to run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config == "cfg5"):
        ap.error("--dump-outputs applies to the TriForce loop of --impl ours (cfg2, cfg3, cfg4)")
    if args.dump_outputs:
        # the split calibrated at start-up follows each SM's measured HBM rate, which varies between processes, and with it the
        # rounding of the attention sums and so the sampled tokens
        os.environ["TRIFORCE_ATTN_CALIBRATE"] = "0"
    if args.config == "cfg3":
        args.target, args.prefill = "lwm-128K", 130048
    elif args.config == "cfg4":
        args.prefill, args.budget, args.gamma = 130048, 12288, 16
    elif args.config == "cfg5":  # Sequoia tree verify (SpecTree_TP, tree/512.pt) on Llama2-13B-128K shapes
        args.target, args.prefill, args.budget = "llama-13B-128K", 131072, 8192
    return args


_T_START = time.time()


def time_left(args, need_s: float) -> bool:
    """Optional legs (acceptance sweep points, the reference on this GPU, the CPU sample, the ncu traffic probe) run only while the
    whole invocation stays inside --time_budget seconds; the timed region and the contract fields never depend on it."""
    return (time.time() - _T_START) + need_s <= args.time_budget


def load_peaks():
    try:
        p = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# Reference arms: the UNMODIFIED reference (baseline/_ref) through baseline/run_reference.py, in a child process
# ---------------------------------------------------------------------------------------------------------------------
def workload_desc(args, weights_desc="random-init fp16 (std 0.02)"):
    return (f"BASELINE {args.config}: {args.target} shapes ({weights_desc}), on-chip, prefill {args.prefill}, budget {args.budget}, "
            f"chunk {args.chunk_size}, gamma {args.gamma}, T {args.temp}, top_p {args.top_p}")


def _mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def ncu_traffic(kv_len: int, heads: int, head_dim: int, rows: int, device_index: int = 0, enabled: bool = True):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel at this line's shape,
    counted NOW: after the timed region rank 0 runs tools/attn_traffic_probe.py (a few launches of tf_verify_attn on fresh keys)
    under `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` and reads the last launch.  DRAM counters cannot be read
    without the profiler; nothing measured under it enters `value` or `roofline.achieved`.  null (with the reason) when ncu is
    not on the box or refuses."""
    import shutil
    import subprocess
    if not enabled:
        return None, "probe disabled (--no_traffic_probe)"
    here = os.path.dirname(os.path.abspath(__file__))
    ncu = shutil.which("ncu") or ("/usr/local/cuda/bin/ncu" if os.path.exists("/usr/local/cuda/bin/ncu") else None)
    if ncu is None:
        return None, "ncu not found on this box"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", "regex:verify_attn_mma_kernel",
           "--launch-skip", "2", "--launch-count", "2", "--csv", sys.executable, os.path.join(here, "tools", "attn_traffic_probe.py"),
           "--kv_len", str(kv_len), "--rows", str(rows), "--heads", str(heads), "--head_dim", str(head_dim), "--device", str(device_index)]
    try:
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    except Exception as e:
        return None, f"ncu probe failed to run: {e!r}"
    import csv as _csv
    rows_ = [x for x in _csv.reader(r.stdout.splitlines()) if len(x) > 8]
    try:
        head = next(i for i, x in enumerate(rows_) if x[0] == "ID")
        col = {n: i for i, n in enumerate(rows_[head])}
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
        per_launch = {}
        for x in rows_[head + 1:]:
            v = float(x[col["Metric Value"]].replace(",", "")) * unit[x[col["Metric Unit"]]]
            per_launch.setdefault(x[col["ID"]], {})[x[col["Metric Name"]]] = v
        last = per_launch[sorted(per_launch, key=int)[-1]]
        total = last["dram__bytes_read.sum"] + last["dram__bytes_write.sum"]
    except Exception as e:
        return None, f"ncu probe gave no counters (rc {r.returncode}): {e!r}; {(r.stderr or r.stdout)[-200:]!r}"
    algo = kv_len * heads * head_dim * 2 * 2
    return total, (f"ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum on tools/attn_traffic_probe.py right after the timed region "
                   f"(kv_len {kv_len}, R {rows}, H {heads}; launch 4 of 4 on alternating layers): read {last['dram__bytes_read.sum']:.0f} B + write "
                   f"{last['dram__bytes_write.sum']:.0f} B = {total / algo:.4f} x the algorithmic bytes")


def run_reference_child(args, device: str, extra, timeout: float) -> dict:
    """baseline/run_reference.py in its own interpreter (its thread count must be set before torch is imported, and the
    reference's `models` / `utils` packages collide with this repo's drop-in packages of the same names)."""
    cmd = [sys.executable, os.path.join(REPO, "baseline", "run_reference.py"), "--device", device, "--target", args.target,
           "--prefill", str(args.prefill), "--budget", str(args.budget), "--chunk_size", str(args.chunk_size), "--gamma", str(args.gamma),
           "--temp", str(args.temp), "--top_p", str(args.top_p), "--seed", str(args.seed)] + [str(x) for x in extra]
    env = {k: v for k, v in os.environ.items()
           if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "MASTER_ADDR", "MASTER_PORT",
                        "OMP_NUM_THREADS", "MKL_NUM_THREADS") and not k.startswith("TORCHELASTIC")}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=REPO)
    except subprocess.TimeoutExpired:
        return {"unavailable": f"baseline/run_reference.py --device {device} exceeded {timeout:.0f} s"}
    for line in reversed(r.stdout.splitlines()):
        if line.startswith("REFERENCE_JSON "):
            return json.loads(line[len("REFERENCE_JSON "):])
    tail = (r.stderr or r.stdout).strip().splitlines()[-1:] or ["no output"]
    return {"unavailable": f"baseline/run_reference.py --device {device} failed (rc {r.returncode}): {tail[0][:300]}"}


def cpu_reference(args, steps: int, warmup: int, timeout: float) -> dict:
    """The reference's CPU HF-eager path on the host cores (kind "reference"): W + K outer TriForce iterations at the bench shapes.
    Host memory: 27 GB of fp32 weights + the fp16 KV store (66 GB at 124 928 keys) — when the box cannot hold that, the KV
    length of the SAMPLE is cut to what fits and said so."""
    from triforce_b200.config import named_config
    cfg = named_config(args.target)
    need = lambda P: (cfg.param_count() * 4 + 2 * cfg.num_hidden_layers * (P + 1100) * cfg.hidden_size * 2) / 1e9 + 14.0
    avail, P = _mem_available_gb(), args.prefill
    note = ""
    while avail and need(P) > avail and P > 8192:
        P //= 2
    if P != args.prefill:
        note = f"; host has {avail:.0f} GB available: KV length of the CPU sample cut from {args.prefill} to {P}"
    sub = argparse.Namespace(**vars(args))
    sub.prefill = P
    r = run_reference_child(sub, "cpu", ["--steps", steps, "--warmup", warmup], timeout)
    if "triforce" not in r:
        return {"error": r.get("unavailable", "no result"), "kind": "reference"}
    t = r["triforce"]
    return dict(value=t["tokens_per_s"], unit=UNIT, cores=int(r.get("threads", 0)), kind="reference", host_cpus=r.get("host_cpus"),
                ms_per_step=t["ms_per_step"], steps=t["steps"], warmup=t["warmup"], tokens_per_step=t["tokens_per_step"],
                seconds=t["seconds"], setup_seconds=r.get("setup_seconds"), prefill_of_sample=P,
                sample=f"the unmodified reference (baseline/_ref: utils/decoding.py::TriForce, torch CPU attention in place of flash-attn, fp32 weights, fp16 KV) on "
                       f"{r.get('threads')} host threads: {t['warmup']} + {t['steps']} outer iterations at {args.target} shapes, budget "
                       f"{args.budget}, gamma {args.gamma}, over a SYNTHETIC {P}-key KV store (the prompt is not prefilled on the CPU), "
                       f"{t['steps']} timed = {t['seconds']:.1f} s{note}")


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return  # under torchrun rank 0 alone runs the CPU arm; the thread count is pinned by the child, identical at every N
    t0 = time.time()
    # one outer iteration of the real loop at the real shapes costs ~11 s on 64 host threads: the sample is bounded to 2 + 10 of them
    # (~2.5 min with set-up) whatever K / W the GPU arm is given; the line reports the counts actually run
    steps, warmup = min(args.steps, 10), min(args.warmup, 2)
    r = cpu_reference(args, steps, warmup, timeout=1500.0)
    if "value" in r and (steps, warmup) != (args.steps, args.warmup):
        r["sample"] += f"; bounded sample: {warmup} + {steps} iterations instead of the requested {args.warmup} + {args.steps}"
    if "value" not in r:
        print(json.dumps({"impl": "reference", "unavailable": r.get("error", "?")}), flush=True)
        return
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"],
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_desc(args),
                       "arm": "the reference's own Python (baseline/_ref) on the host CPU cores: fp32 weights, fp16 KV, torch's fused CPU "
                              "attention in place of flash-attn, eager callables in place of CUDA graphs — no CUDA"},
            "tokens_per_step": r["tokens_per_step"], "cpu_baseline": r, "gpu_launches": 0, "wall_seconds": time.time() - t0,
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    with open(REFERENCE_LAST, "w") as f:
        json.dump(dict(line, when=time.time(), args=dict(target=args.target, prefill=args.prefill, budget=args.budget, gamma=args.gamma)), f)
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def dump_outputs(out_dir: str, run, produced: int, loop: str) -> None:
    """--dump-outputs: the tokens the last timed step handed back to its caller, and the target's probabilities over the vocabulary
    at the rows that step verified over the full KV (the distribution its tokens were accepted against or resampled from)."""
    import numpy as np
    tokens = run.generated[len(run.generated) - produced:]
    probs = run.loop.full_probs[:run.records[-1][3] + 1] if loop == "device" else run.full_probs
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tokens.npy"), np.asarray(tokens, dtype=np.float64))
    np.save(os.path.join(out_dir, "target_probs.npy"), probs.float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    from triforce_b200 import ops
    from triforce_b200.cache import FlashSimpleCache, RetrievalCache, StreamingLLMEvictionCache
    from triforce_b200.config import named_config
    from triforce_b200.decoding import TriForceRun, _sample_token
    from triforce_b200.device_loop import DeviceLoopRun
    from triforce_b200.engine import GraphInferenceEngine
    from triforce_b200.llama import LlamaModel
    from triforce_b200.rng import TorchNoise
    from triforce_b200.sampling import norm_logits
    from triforce_b200.synth import cuda_state_dict

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # keep stdout to rank 0's one JSON line: NCCL prints "NCCL version ..." (and any debug output) to stdout by default
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    torch.manual_seed(args.seed)  # every rank: identical sampling streams replace the reference's broadcast+barrier

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg_t, cfg_d = named_config(args.target), named_config("llama-68M")
    gamma, P = args.gamma, args.prefill
    if args.weights.startswith("agreement:"):
        from triforce_b200.synth import agreement_state_dicts
        a_t, a_d = (float(x) for x in args.weights.split(":")[1].split(","))
        tsd, dsd = agreement_state_dicts(cfg_t, cfg_d, a_t, a_d, seed=0, device=dev)
        weights_desc = f"acceptance-calibrated synthetic (shared token table, layer outputs x{a_t} target / x{a_d} draft)"
    else:
        tsd, dsd = cuda_state_dict(cfg_t, seed=1, device=dev), cuda_state_dict(cfg_d, seed=2, device=dev)
        weights_desc = "random-init fp16 (std 0.02)"
    target = LlamaModel(cfg_t, tsd, device=dev, tp_rank=rank, tp_world=world)
    target.attn_variant = args.attn_variant
    if world > 1:
        t = torch.zeros(8, device=dev)
        dist.all_reduce(t)  # create the NCCL communicator before any CUDA-graph capture
        target.enable_peer_allreduce()
    draft = LlamaModel(cfg_d, dsd, device=dev, is_draft=True)
    del tsd, dsd
    torch.cuda.empty_cache()
    # KV slots past the prompt: --gen_len, or more when the steps of one run (warm-up, timed, e2e) could outgrow it by accepting
    # every draft, so that --steps K runs K steps whatever K is
    reserve = max(args.gen_len, (args.warmup + 2 * max(args.steps, args.sweep_steps)) * (gamma + 1) + gamma + 2)
    cache = FlashSimpleCache(target, P + reserve + 16)
    graph_cache = RetrievalCache(target, max_budget=args.budget, prefill=P, gamma=gamma, chunk_size=args.chunk_size)
    draft_cache = StreamingLLMEvictionCache(draft, start_size=16, recent_size=256 - 16 - gamma, gamma=gamma)
    ge = GraphInferenceEngine(target, cache, graph_cache, draft, draft_cache)
    ge.engine.target_prefill_chunk = args.prefill_chunk
    ge.initialize_cuda_graph(gamma, probs=True, temperature=args.temp, top_p=args.top_p)

    # synthetic prompt: pinned host buffer → device (the step inputs of the e2e leg come from pinned memory as well)
    g = torch.Generator().manual_seed(args.seed)
    prompt_host = torch.randint(0, cfg_t.vocab_size, (1, P), generator=g).pin_memory()
    input_ids = prompt_host.to(dev, non_blocking=True)

    tok = type("Tok", (), {"eos_token_id": 2, "decode": lambda self, *a, **k: ""})()
    noise = TorchNoise(dev)
    t_setup = time.time()

    # ---- prefill (untimed, like the reference) + autoregressive baseline ---------------------------------------------
    with torch.inference_mode():
        cache.reset()
        logits = ge.inference(input_ids=input_ids)
        torch.cuda.synchronize()
        prefill_s = time.time() - t_setup
        buf_expo = torch.empty(cfg_t.vocab_size, dtype=torch.float32, device=dev)
        nxt = _sample_token(norm_logits(logits[:, -1, :], temperature=args.temp, top_k=-1, top_p=args.top_p), noise, buf_expo)

        def ar_step(tk):
            lg = ge.decode_step(tk)
            return _sample_token(norm_logits(lg[:, -1, :], temperature=args.temp, top_k=-1, top_p=args.top_p), noise, buf_expo)

        for _ in range(max(args.warmup, 3)):
            nxt = ar_step(nxt)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.ar_steps):
            nxt = ar_step(nxt)
        e1.record()
        barrier()
        ar_ms = e0.elapsed_time(e1) / args.ar_steps

        # ---- TriForce: rebuild the hierarchy on the same prompt KV, warm up, then time exactly K steps ------------------
        def make_run():
            if args.loop == "device":
                return DeviceLoopRun(tok, ge, gamma=gamma, top_p=args.top_p, temperature=args.temp, seed=args.seed, max_new=args.gen_len)
            return TriForceRun(tok, ge, gamma=gamma, top_p=args.top_p, temperature=args.temp, noise=noise)

        def e2e_step(r):
            """One step through the public step API with HOST buffers: the step's input token comes from pinned host memory, its
            result tokens go back to pinned host memory (the device loop reads its result record back by construction)."""
            host_in[0] = r.next_token
            if args.loop == "device":
                r.loop.first_token.copy_(host_in[:1], non_blocking=True)   # step input: host → device
                r.step()                                                   # result record + tokens: device → pinned host
            else:
                dev_in.copy_(host_in, non_blocking=True)
                r.next_token = int(dev_in[0].item())
                r.step()
                host_out.copy_(r.buf.pass_tokens[0], non_blocking=True)
                torch.cuda.current_stream().synchronize()

        run = make_run()
        run.prefill(input_ids, skip_target_prefill=True)
        for _ in range(args.warmup):
            run.step()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        n0, inner0, launches0 = run.n, run.inner_iterations, ops.COUNTER.n
        acc0, dr0 = run.accepted_count, run.draft_count
        barrier()
        profiling = os.environ.get("TF_PROFILE") == "1"  # ncu --profile-from-start off: capture the timed steps only
        if profiling:
            torch.cuda.profiler.start()
        w0 = time.time()
        e0.record()
        for _ in range(args.steps):
            produced = run.step()
        e1.record()
        barrier()
        w1 = time.time()
        if profiling:
            torch.cuda.profiler.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, run, produced, args.loop)
        dev_ms = e0.elapsed_time(e1)
        tokens = run.n - n0
        inner = run.inner_iterations - inner0
        launches = ops.COUNTER.n - launches0
        acc_rate = (run.accepted_count - acc0) / max(run.draft_count - dr0, 1)
        clocks = sampler.stop(w0, w1) if rank == 0 else None
        if world > 1:
            t = torch.tensor([dev_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dev_ms = float(t.item())

        # ---- e2e leg: the same K steps through the public step API with HOST buffers ------------------------------------
        # every step copies its input token ids from pinned host memory and reads its result tokens back to the host
        host_in = torch.zeros(gamma + 2, dtype=torch.int64).pin_memory()
        host_out = torch.zeros(gamma + 3, dtype=torch.int64).pin_memory()
        dev_in = torch.zeros(gamma + 2, dtype=torch.int64, device=dev)
        h2d = d2h = 0
        n1 = run.n
        b0, d0 = run.h2d_bytes, run.d2h_bytes
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step(run)
            h2d += 8 if args.loop == "device" else host_in.numel() * 8
            d2h += 0 if args.loop == "device" else host_out.numel() * 8
        barrier()
        t1 = time.perf_counter()
        e2e_tokens = run.n - n1
        e2e_s = t1 - t0
        if world > 1:
            t = torch.tensor([e2e_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        h2d += run.h2d_bytes - b0
        d2h += run.d2h_bytes - d0

        # ---- roofline of the dominant kernel (full-KV verify attention), measured live with CUDA events ----------------
        Hl, d = target.local_num_heads, target.head_dim
        outer_steps = run.steps if args.loop == "device" else len(run.acc_rate_middle_list)
        R = (gamma + 2) if args.loop == "device" else max(2, round((run.draft_count / max(outer_steps, 1)) + 1))
        kv_len = cache.seq_len + R
        q = torch.randn((R, Hl, d), device=dev, dtype=torch.float16)
        o = torch.empty_like(q)
        ws = target._workspace()
        L = cfg_t.num_hidden_layers
        for l in range(3):
            ops.verify_attn(q, cache.tensor_maps, l, kv_len, R, Hl, d, target.scale, o, ws, variant=args.attn_variant)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(L)]
        torch.cuda.synchronize()
        for l, (a, b) in enumerate(evs):  # one launch per layer: 2 GB of distinct KV each, far beyond the 126 MB L2
            a.record()
            ops.verify_attn(q, cache.tensor_maps, l, kv_len, R, Hl, d, target.scale, o, ws, variant=args.attn_variant)
            b.record()
        torch.cuda.synchronize()
        attn_ms = sum(a.elapsed_time(b) for a, b in evs) / L
        attn_bytes = kv_len * Hl * d * 2 * 2
        peak, peak_src = load_peaks()
        achieved = attn_bytes / (attn_ms * 1e-3) / 1e9
        traffic, traffic_src = (None, "counted by an ncu child process after the timed region at N = 1 only")

        # ---- the other half of the step's device time (profiles/r02_launch_list_final.md: 53 %): tf_stream_linear, EVERY projection
        #      of one R-row target forward (q|k|v, o_proj, gate|up + SiLU·mul, down_proj per layer, lm_head) as one CUDA graph,
        #      timed with CUDA events; bytes = the weights it streams (distinct per layer, 13 GB >> L2) ---------------------------
        proj = None
        try:
            lws = target.layers
            if target.use_stream_linear and all(w.m_qkv and w.m_o and w.m_gu and w.m_d for w in lws) and target.m_lm_head is not None:
                xr = torch.randn((R, cfg_t.hidden_size), device=dev, dtype=torch.float16)
                xo = torch.randn((R, lws[0].m_o.K), device=dev, dtype=torch.float16)
                xd = torch.zeros((R, lws[0].m_d.K), device=dev, dtype=torch.float16)
                lws_ws = target._linear_ws

                def all_projections():
                    for w in lws:
                        ops.stream_linear(xr, w.m_qkv, workspace=lws_ws)
                        ops.stream_linear(xo, w.m_o, workspace=lws_ws)
                        ops.stream_linear(xr, w.m_gu, silu=True, workspace=lws_ws)
                        ops.stream_linear(xd, w.m_d, workspace=lws_ws)
                    ops.stream_linear(xr, target.m_lm_head, out_fp32=True, workspace=lws_ws)

                n0_launch = ops.COUNTER.n
                all_projections()
                torch.cuda.synchronize()
                gproj = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gproj):
                    all_projections()
                ops.COUNTER.n = n0_launch  # a side measurement: not part of the step's launch count
                for _ in range(3):
                    gproj.replay()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(10):
                    gproj.replay()
                e1.record()
                torch.cuda.synchronize()
                proj_ms = e0.elapsed_time(e1) / 10
                proj_bytes = 2 * (sum(w.m_qkv.N * w.m_qkv.K + w.m_o.N * w.m_o.K + w.m_gu.N * w.m_gu.K + w.m_d.N * w.m_d.K for w in lws)
                                  + target.m_lm_head.N * target.m_lm_head.K)
                proj = {"kernel": "stream_linear_kernel<1> (every projection of one target forward)", "bound": "hbm", "rows": R,
                        "launches": 4 * len(lws) + 1, "bytes": proj_bytes, "ms": proj_ms, "achieved": proj_bytes / (proj_ms * 1e-3) / 1e9,
                        "peak": peak, "unit": "GB/s", "frac": proj_bytes / (proj_ms * 1e-3) / 1e9 / peak,
                        "how": "CUDA events around 10 replays of one CUDA graph holding the launches (PDL-chained), same process, after the "
                               "timed steps; algorithmic bytes = N*K*2 B of weights per launch"}
                del gproj
        except Exception as e:  # a side measurement must never take the line down
            proj = {"error": repr(e)[:200]}

        # ---- the kernel to beat (SURVEY §2b K1): flash-attn's FA2 through the reference's own call (modeling_llama.py:240), on
        #      keys of the same count in the reference's [S,H,d] layout, timed the same way right here -------------------------
        vs_fa2 = None
        if rank == 0:
            try:
                from flash_attn import flash_attn_with_kvcache
                nbuf = 3
                Kr = torch.randn((nbuf, 1, kv_len, Hl, d), device=dev, dtype=torch.float16)
                Vr = torch.randn((nbuf, 1, kv_len, Hl, d), device=dev, dtype=torch.float16)
                qr = q[None].contiguous()
                for i in range(3):
                    flash_attn_with_kvcache(qr, Kr[i % nbuf], Vr[i % nbuf], softmax_scale=target.scale, causal=True)
                fe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(12)]
                torch.cuda.synchronize()
                for i, (a, b) in enumerate(fe):
                    a.record()
                    flash_attn_with_kvcache(qr, Kr[i % nbuf], Vr[i % nbuf], softmax_scale=target.scale, causal=True)
                    b.record()
                torch.cuda.synchronize()
                fa_ms = sum(a.elapsed_time(b) for a, b in fe) / len(fe)
                vs_fa2 = {"fa2_ms_per_launch": fa_ms, "fa2_gbs": attn_bytes / (fa_ms * 1e-3) / 1e9, "fa2_frac_of_peak": attn_bytes / (fa_ms * 1e-3) / 1e9 / peak,
                          "ours_over_fa2": fa_ms / attn_ms,
                          "how": f"flash_attn_with_kvcache (flash-attn FA2 sm_100 cubin) q [1,{R},{Hl},{d}] over k/v [1,{kv_len},{Hl},{d}], "
                                 "causal, CUDA events around 12 eager launches over 3 rotating KV buffers"}
                del Kr, Vr
            except Exception as e:
                vs_fa2 = {"unavailable": repr(e)[:200]}

        # ---- acceptance sweep: the same job, kernels and bytes on acceptance-calibrated synthetic weights (synth.py) --------
        sweep = []
        if world == 1 and args.sweep and args.weights == "random":
            from triforce_b200.synth import retune_agreement
            state = {"alpha_t": 1.0, "alpha_d": 1.0, "shared_table": False}
            for alpha in [float(a) for a in args.sweep.split(",") if a.strip() != ""]:
                if not time_left(args, 30.0 + 300.0):  # keep room for the reference-on-this-GPU leg and the probe
                    sweep.append({"alpha": alpha, "skipped": "time budget"})
                    continue
                retune_agreement(target, draft, alpha, alpha, state)
                cache.reset()
                ts = time.time()
                ge.inference(input_ids=input_ids)  # the prompt KV belongs to the weights: prefill again (untimed)
                run = make_run()
                run.prefill(input_ids, skip_target_prefill=True)
                for _ in range(args.warmup):
                    run.step()
                torch.cuda.synchronize()
                n0, i0, a0, d0 = run.n, run.inner_iterations, run.accepted_count, run.draft_count
                e0.record()
                for _ in range(args.sweep_steps):
                    run.step()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                toks = run.n - n0
                acc_sw = (run.accepted_count - a0) / max(run.draft_count - d0, 1)
                inner_sw = (run.inner_iterations - i0) / args.sweep_steps
                n1 = run.n
                t0 = time.perf_counter()
                for _ in range(args.sweep_steps):  # e2e: step input from pinned host memory, result tokens back to the host
                    e2e_step(run)
                e2e_sw = (run.n - n1) / (time.perf_counter() - t0)
                tps = toks / (ms * 1e-3)
                sweep.append({"alpha": alpha, "acceptance_rate": acc_sw,
                              "tokens_per_step": toks / args.sweep_steps, "inner_per_step": inner_sw,
                              "ms_per_step": ms / args.sweep_steps, "tokens_per_s": tps, "e2e_tokens_per_s": e2e_sw,
                              "ar_tokens_per_s": 1000.0 / ar_ms, "speedup_vs_ar": tps / (1000.0 / ar_ms),
                              "e2e_speedup_vs_ar": e2e_sw / (1000.0 / ar_ms), "steps": args.sweep_steps, "prefill_seconds": None})
                sweep[-1]["prefill_seconds"] = round(time.time() - ts - ms * 1e-3, 1)

    if rank != 0:
        _finish(world)
        return
    steps = args.steps
    value = tokens / (dev_ms * 1e-3)
    ar_tps = 1000.0 / ar_ms
    tokens_per_step = tokens / steps
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic",
        "config": {"workload": workload_desc(args, weights_desc),
                   "parallelism": (f"tp{world} (head-sharded; all-reduce on the o_proj/down_proj seams: " + (
                                   f"fused into the seam GEMV (tf_stream_linear_allreduce over {target.peer_stream.transport})" if getattr(target, "peer_stream", None)
                                   else f"this library's NVLink exchange over {target.peer_allreduce.transport}" if target.peer_allreduce else "NCCL") + ")")
                   if world > 1 else "single GPU",
                   "l2": "no flush needed: every step streams 79 GB (KV 65.5 GB + weights 13.5 GB per target forward) >> 126 MB L2",
                   "kv_layout": "head-major [L,H,S,d] fp16", "step": "one TriForce outer iteration"},
        "weights": weights_desc,
        "ms_per_token": dev_ms / max(tokens, 1),
        "tokens_per_step": tokens_per_step,
        "avg_accepted_len": acc_rate * gamma,
        "acceptance_rate": acc_rate,
        "inner_per_step": inner / steps,
        "rows_full_verify": R,
        "ar_baseline": {"tokens_per_s": ar_tps, "ms_per_token": ar_ms, "steps": args.ar_steps,
                        "how": "full-KV decode step as one CUDA graph + fused sampling (the reference runs it eagerly)"},
        "speedup_vs_ar": value / ar_tps,
        "e2e": {"value": e2e_tokens / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d / steps, "d2h_bytes_per_step": d2h / steps,
                # the e2e loop times the NEXT K steps of the same run: with random-init weights the tokens a step yields vary
                # (1.0-1.25), so compare the per-step times, not only the rates
                "ms_per_step": e2e_s * 1e3 / steps, "tokens_per_step": e2e_tokens / steps, "steps": steps,
                "how": ("DeviceLoopRun.step(): the step's input token copied from pinned host memory, ONE graph launch, the result record "
                        "(counts + tokens) copied back to pinned host memory by the graph itself" if args.loop == "device" else
                        "TriForceRun.step() with the step's token ids copied from pinned host memory and the result tokens read "
                        "back to pinned host memory") + " — inside the timed region (wall clock, synchronised both sides)"},
        "loop": ("device: one CUDA-graph launch per outer step, Middle_Spec = conditional WHILE node, one host read-back per step"
                 if args.loop == "device" else "host: step-wise loop, one host synchronisation per inner iteration"),
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": "verify_attn_mma_kernel (full-KV verify attention)", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "vs_fa2": vs_fa2,
                     "projections": proj,
                     "bytes_per_launch": attn_bytes, "ms_per_launch": attn_ms,
                     "how": f"CUDA events around {L} eager launches (one per layer, R={R}, kv_len={kv_len}) on the launching stream, "
                            "same process, right after the timed steps; algorithmic bytes = kv_len*H*d*2(K,V)*2 B",
                     "frac_of_nominal_8TBs": achieved / 8000.0,
                     "note": "the peak is the measured COPY bandwidth (reads + writes); a read-only stream can exceed it, so frac may be > 1",
                     "split_calibration": getattr(target, "attn_balance", None)},
        "clocks": clocks,
        "prefill_seconds": prefill_s,
        "acceptance_sweep": {"points": sweep,
                             "how": "synth.retune_agreement: draft and target share one token table and every layer's o_proj / down_proj is "
                                    "scaled by alpha (alpha = 1: unrelated random models; alpha = 0: the three levels agree); shapes, kernels "
                                    "and bytes per forward are unchanged; the prompt is prefilled again for every alpha; AR is the line's "
                                    "ar_baseline (weight values do not change its speed)"} if sweep else None,
    }
    if world == 1:
        # free the engine (80 GB) before the reference legs run in child processes
        del run, ge, cache, graph_cache, draft_cache, target, draft, q, o, ws
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        # DRAM bytes of one launch of the roofline kernel at this line's shape, counted by ncu in a child process (after, and
        # outside, every timed region)
        tr, tr_src = ncu_traffic(kv_len, Hl, d, R, device_index=dev.index or 0, enabled=not args.no_traffic_probe) if time_left(args, 60.0) \
            else (None, "skipped: time budget")
        line["roofline"]["traffic"], line["roofline"]["traffic_source"] = tr, tr_src
        if not args.no_reference_gpu and not time_left(args, 170.0):
            line["reference_gpu"] = {"unavailable": "skipped: time budget"}
        elif not args.no_reference_gpu:
            try:
                line["reference_gpu"] = run_reference_child(args, "cuda", ["--gen_len", 96, "--ar_len", 32, "--warmup_calls", 1],
                                                            timeout=args.reference_gpu_timeout)
                rg = line["reference_gpu"]
                if "triforce" in rg:
                    line["vs_reference_gpu"] = {"tokens_per_s_ratio": value / rg["triforce"]["tokens_per_s"],
                                                "ar_ms_per_token_ratio": rg["autoregressive"]["ms_per_token"] / ar_ms,
                                                "note": "ours / the reference with real flash-attn on the same B200, same shapes, weights and prompt"}
            except Exception as e:
                line["reference_gpu"] = {"unavailable": repr(e)[:300]}
        if not args.no_cpu_baseline:
            try:  # a `--impl reference` run on this host shortly before: reuse its measurement, else take a short sample
                last = json.load(open(REFERENCE_LAST))
                same = last["args"] == dict(target=args.target, prefill=args.prefill, budget=args.budget, gamma=args.gamma)
                if same and time.time() - last["when"] < 7200 and time.time() - last["when"] < _uptime_seconds():
                    line["cpu_baseline"] = dict(last["cpu_baseline"], reused="measured by `bench.py --impl reference` on this box "
                                                f"{time.time() - last['when']:.0f} s earlier")
            except Exception:
                pass
            if "cpu_baseline" not in line and not time_left(args, 120.0):
                line["cpu_baseline"] = {"error": "skipped: time budget (run `bench.py --impl reference`)", "kind": "reference"}
            if "cpu_baseline" not in line:
                try:
                    line["cpu_baseline"] = cpu_reference(args, steps=3, warmup=1, timeout=900.0)
                except Exception as e:  # the CPU leg must never take the GPU number down with it
                    line["cpu_baseline"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    _finish(world)


def run_cfg5(args):
    """BASELINE cfg5: Llama2-13B-128K shapes, prefill 128K, retrieval budget 8192, the 512-node Sequoia tree (utils/SpecTree_TP.py,
    test/offloading_seqouia.py:148-205).  A STEP = grow the tree over the retrieval cache (16 masked forwards) + ONE masked verify of
    all 512 nodes over the full KV (tcgen05 attention, tf_tree_attn_tc) + accept walk + KV compaction.  Single GPU."""
    import torch

    from triforce_b200 import ops
    from triforce_b200.spectree import SpecTree, get_residual, load_grow_map
    from triforce_b200.synth import cuda_state_dict
    from triforce_b200.tp import DistributedLlama

    assert int(os.environ.get("WORLD_SIZE", "1")) == 1, "cfg5 is benchmarked on one GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    torch.manual_seed(args.seed)
    grow_map = load_grow_map(args.tree_size)
    T = grow_map["size"]
    llm = DistributedLlama(model_name_or_path=args.target, local_rank=0, world_size=1, prefill=args.prefill, gen_len=args.gen_len,
                           temperature=args.temp, top_p=args.top_p, retrieval_budget=args.budget, retrieval_chunk_size=args.chunk_size,
                           tree_size=T)
    llm.init_parameters(state_dict=cuda_state_dict(llm.config, seed=1, device=dev), cuda_graphs=False)
    tok = type("Tok", (), {"eos_token_id": 2, "decode": lambda self, *a, **k: ""})()
    tree = SpecTree(engine=llm, temperature=args.temp, top_p=args.top_p, max_length=args.prefill + args.gen_len, grow_map=grow_map,
                    residual_graph=get_residual, tokenizer=tok, vocab_size=llm.config.vocab_size)
    g = torch.Generator().manual_seed(args.seed)
    ids = torch.randint(0, llm.config.vocab_size, (args.prefill,), generator=g).pin_memory().to(dev, non_blocking=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.inference_mode():
        t0 = time.time()
        next_token = tree.prefill(prefix=ids)
        torch.cuda.synchronize()
        prefill_s = time.time() - t0
        # autoregressive baseline at the same geometry (eager one-row forwards over the full KV), then roll the cache back
        seq0 = llm.kv_cache.seq_len
        nt = next_token.reshape(1, 1)
        for _ in range(2):
            llm.inference(input_ids=nt)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.ar_steps):
            llm.inference(input_ids=nt)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / args.ar_steps
        llm.kv_cache.seq_len = seq0

        def step(tokn):
            tree.construct_grow_map(next_token=tokn)
            nxt, acc, _ = tree.verify()
            if nxt is None:  # an EOS id was accepted: keep the benchmark going from a fixed token
                nxt = torch.full((1,), 5, dtype=torch.long, device=dev)
            return nxt.unsqueeze(0), acc

        for _ in range(args.warmup):
            next_token, _ = step(next_token)
        torch.cuda.synchronize()
        sampler = ClockSampler(0)
        sampler.start()
        time.sleep(0.25)
        launches0 = ops.COUNTER.n
        w0 = time.time()
        tokens = 0
        e0.record()
        for _ in range(args.steps):
            next_token, acc = step(next_token)
            tokens += acc
        e1.record()
        torch.cuda.synchronize()
        w1 = time.time()
        dev_ms = e0.elapsed_time(e1)
        launches = ops.COUNTER.n - launches0
        clocks = sampler.stop(w0, w1)
        # e2e: the step's first token comes from pinned host memory, the accepted tokens go back to pinned host memory
        host_in = torch.zeros(1, dtype=torch.int64).pin_memory()
        host_out = torch.zeros(32, dtype=torch.int64).pin_memory()
        dev_in = torch.zeros((1, 1), dtype=torch.int64, device=dev)
        e2e_tokens = 0
        t0 = time.perf_counter()
        for _ in range(args.steps):
            host_in[0] = int(next_token.reshape(-1)[0].item())
            dev_in.copy_(host_in.view(1, 1), non_blocking=True)
            next_token, acc = step(dev_in.clone())
            host_out[:1].copy_(next_token.reshape(-1)[:1], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            e2e_tokens += acc
        e2e_s = time.perf_counter() - t0
        # roofline of the dominant kernel: the 512-row tree verify attention on the tensor cores
        m = llm.model
        Hl, d = m.local_num_heads, m.head_dim
        kv_len = llm.kv_cache.seq_len + T
        q = torch.randn((T, Hl, d), device=dev, dtype=torch.float16)
        o = torch.empty_like(q)
        ws = ops.tree_attn_tc_workspace(T, Hl, int(llm.kv_cache.tensor_maps.shape[2]), dev)
        for l in range(2):
            ops.tree_attn_tc(q, llm.kv_cache.tensor_maps, l, kv_len, T, Hl, d, m.scale, tree.mask_bits, T, o, ws)
        L = min(8, llm.config.num_hidden_layers)
        torch.cuda.synchronize()
        e0.record()
        for l in range(L):
            ops.tree_attn_tc(q, llm.kv_cache.tensor_maps, l, kv_len, T, Hl, d, m.scale, tree.mask_bits, T, o, ws)
        e1.record()
        torch.cuda.synchronize()
        attn_ms = e0.elapsed_time(e1) / L
        flops = 4.0 * T * kv_len * Hl * d
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        peak_tf, peak_src = float(peaks["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"
    achieved = flops / (attn_ms * 1e-3) / 1e12
    value = tokens / (dev_ms * 1e-3)
    line = {"metric": "decode tokens/sec at 128K prefill (Sequoia tree 512 over the retrieval cache, Llama2-13B-128K shapes, budget 8192)",
            "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": workload_desc(args) + f", tree {T} (tree/512.pt topology)", "parallelism": "single GPU",
                       "step": "grow the 512-node tree (16 masked forwards over the retrieval cache) + one masked 512-row verify over the full KV"},
            "tokens_per_step": tokens / args.steps, "ms_per_token": dev_ms / max(tokens, 1),
            "ar_baseline": {"tokens_per_s": 1000.0 / ar_ms, "ms_per_token": ar_ms, "steps": args.ar_steps, "how": "eager one-row full-KV forwards"},
            "speedup_vs_ar": value / (1000.0 / ar_ms),
            "e2e": {"value": e2e_tokens / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 8, "d2h_bytes_per_step": 8 + 128,
                    "how": "step input token from pinned host memory, accepted-token read-back to the host inside the timed region"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "tree_attn_tc_kernel (tcgen05 512-row tree verify attention)", "achieved": achieved,
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "peak_source": peak_src, "traffic": None,
                         "flops_per_launch": flops, "ms_per_launch": attn_ms,
                         "how": f"CUDA events around {L} launches (one per layer, {T} rows x {kv_len} keys x {Hl} heads); algorithmic FLOP = 4*R*S*H*d"},
            "clocks": clocks, "prefill_seconds": prefill_s}
    print(json.dumps(line), flush=True)


def _uptime_seconds() -> float:
    try:
        return float(open("/proc/uptime").read().split()[0])
    except Exception:
        return 1e12


def _finish(world):
    """Multi-rank teardown: NCCL communicators captured inside CUDA graphs can stall interpreter shutdown, so flush and
    leave without running destructors (everything that matters has been printed)."""
    if world > 1:
        import torch.distributed as dist
        try:
            dist.barrier()
        except Exception:
            pass
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.config == "cfg5":
        run_cfg5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
