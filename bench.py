#!/usr/bin/env python
"""bench.py — tokens/s + acceptance rate of self-speculative decoding (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A STEP is one full generation: a 128-id synthetic prompt -> a 512-token greedy continuation,
Llama-2-7B architecture, random-init weights (seeded), exit_layer 8, num_speculations 6 —
BASELINE.json `configs[1]`.  Prefill is inside the timed region, exactly as the reference
times it (self_speculation/generator_base.py:107-129).

  value  : total generated tokens / device time (CUDA events on the engine's stream around
           prefill and every round), inputs already resident on the device.
  e2e    : the same generations timed by wall clock through the reference-facing plug-in call
           `B200SelfSpeculativeGenerationStrategy.generate_token_ids` — host prompt ids in, host
           token ids out, every host<->device copy and the per-round sync inside the region.
  N > 1  : one process per GPU (torchrun).  The path is batch-1 decoding, so ranks are
           independent replicas serving different prompts (weak scaling, no data-path
           collective); `--tp` instead shards ONE model tensor-parallel over the N GPUs.
  --dump-outputs DIR : after the timed steps, what the last timed generation returned (tokens,
           acceptance, per-round results) as DIR/<name>.npy.  Weights and prompts are seeded, so
           runs with the same arguments see the same inputs and two builds compare output for output.

`--impl reference` times the reference algorithm's CPU implementation (the oracle port of
/root/reference/self_speculation/*, which cannot travel to the GPU box) on the host cores, on a
bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tokens_per_second_self_speculative_greedy"
UNIT = "tokens/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arch", default="llama2-7b")
    ap.add_argument("--exit-layer", type=int, default=8)
    ap.add_argument("--num-speculations", type=int, default=6)
    ap.add_argument("--prompt-len", type=int, default=128)
    ap.add_argument("--max-steps", type=int, default=512)
    ap.add_argument("--alpha", type=float, default=1.0,
                    help="late-layer damping of the synthetic model (1.0 = pure random init)")
    ap.add_argument("--tp", action="store_true", help="(default for N > 1) tensor-parallel over the N GPUs")
    ap.add_argument("--replicas", action="store_true",
                    help="N > 1: make the independent-replicas leg the headline instead of tensor parallelism")
    ap.add_argument("--deadline", type=float, default=800.0,
                    help="seconds after which the watchdog prints the best line it has and exits")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the acceptance sweep / AR legs")
    ap.add_argument("--cpu-max-steps", type=int, default=0, help="reference arm: tokens per step")
    ap.add_argument("--cpu-budget", type=float, default=300.0,
                    help="reference arm: seconds of CPU time the K timed generations may take in total")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed generation returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the engine arm (--impl b200)")
    return args


# --------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.QUERY}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return float(json.load(f)["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


# --------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------------
def usable_cpus() -> int:
    """CPUs this process may really use: affinity mask, capped by the cgroup CPU quota (a box
    can show 128 cores while the container is throttled to far fewer — running 128 OpenMP
    threads there is two orders of magnitude slower than running 16)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
        except Exception:
            pass
    return max(1, n)


CPU_THREADS = None


def cpu_threads() -> int:
    global CPU_THREADS
    if CPU_THREADS is None:
        CPU_THREADS = min(32, usable_cpus())     # batch-1 GEMV is DRAM-bound: 32 threads saturate it
    return CPU_THREADS


class time_limit:
    """Hard wall-clock bound for the CPU legs (SIGALRM -> TimeoutError between torch ops)."""

    def __init__(self, seconds):
        self.seconds = int(seconds)

    def __enter__(self):
        import signal

        def handler(signum, frame):
            raise TimeoutError(f"CPU leg exceeded {self.seconds} s")
        self.old = signal.signal(signal.SIGALRM, handler)
        signal.alarm(self.seconds)

    def __exit__(self, *exc):
        import signal
        signal.alarm(0)
        signal.signal(signal.SIGALRM, self.old)
        return False


def cpu_weights(sd, arch):
    """Oracle weights on the host: fp32 when RAM allows (torch's CPU bf16 matmul is an order of
    magnitude slower than fp32 on these Xeons), else bf16."""
    import psutil
    import torch
    from oracle import llama_oracle as orc
    dims = orc.LlamaDims(vocab=arch.vocab, hidden=arch.hidden, inter=arch.inter,
                         layers=arch.layers, heads=arch.heads, kv_heads=arch.kv_heads,
                         head_dim=arch.head_dim, rms_eps=arch.rms_eps, rope_theta=arch.rope_theta)
    need_fp32 = 2 * arch.param_bytes()
    dtype = torch.float32 if psutil.virtual_memory().available > 1.5 * need_fp32 else torch.bfloat16
    return orc.weights_from_state_dict(dims, sd, dtype=dtype), str(dtype).replace("torch.", "")


def cpu_reference_run(args, w, arch, prompts, n_generations, max_steps):
    """Time `n_generations` greedy self-speculative generations of `max_steps` tokens with the
    oracle (CPU restatement of the reference algorithm).  Returns (tokens, seconds, acc)."""
    import torch
    from oracle import llama_oracle as orc
    torch.set_num_threads(cpu_threads())
    tokens, seconds, rates = 0, 0.0, []
    with torch.inference_mode():
        for i in range(n_generations):
            prompt = prompts[i % len(prompts)]
            t0 = time.perf_counter()
            res = orc.self_speculative_generate(
                w, prompt, [arch.vocab - 1], max_steps=max_steps, exit_layer=args.exit_layer,
                num_speculations=args.num_speculations, sample=False)
            seconds += time.perf_counter() - t0
            tokens += len(res.predicted_tokens)
            rates.append(res.acceptance_rate)
    return tokens, seconds, sum(rates) / max(1, len(rates))


def cpu_probe(args, w, arch, prompts):
    """Prefill cost and per-round cost of the CPU implementation, from two short generations
    (2 and 6 tokens): seconds(n) = prefill + rounds(n) * per_round.  Doubles as warm-up."""
    t0 = time.perf_counter()
    cpu_reference_run(args, w, arch, prompts, 1, 2)
    t2 = time.perf_counter() - t0
    t0 = time.perf_counter()
    cpu_reference_run(args, w, arch, prompts, 1, 6)
    t6 = time.perf_counter() - t0
    per_round = max((t6 - t2) / 4.0, 1e-4)             # acceptance ~0 on random init: 1 token per round
    prefill = max(t2 - 2 * per_round, 0.0)
    return prefill, per_round, t2 + t6


def cpu_sized_sample(args, w, arch, prompts, budget_s):
    """Continuation length so that ONE generation costs about `budget_s` of CPU time, between 16
    tokens (below that the prefill dominates the rate) and 64."""
    prefill, per_round, spent = cpu_probe(args, w, arch, prompts)
    n = int(max(16, min(64, (budget_s - prefill) / per_round)))
    return n, spent, prefill, per_round


def tp_collectives_name():
    return {"0": "nccl all-reduce + residual add",
            "1": "peer one-shot LL kernel after the GEMM (csrc/tp_peer.cuh)",
            "3": "peer one-shot, fence + flag protocol"}.get(
                os.environ.get("LSK_TP_ONESHOT", "2"),
                "row-parallel GEMM pushes LL lines to every rank from its epilogue + poll/sum kernel "
                "(csrc/gemm_skinny.cuh EPI_PUSH, csrc/tp_peer.cuh)")


def workload_string(args):
    return (f"{args.arch} arch, random-init (alpha={args.alpha}), exit_layer={args.exit_layer}, "
            f"num_speculations={args.num_speculations}, greedy, {args.prompt_len}-id synthetic prompts, "
            f"{args.max_steps}-token continuations")


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from layerskip_b200.synthetic import synthetic_prompts
    from layerskip_b200.weights import ARCHS, SyntheticLlama
    arch = ARCHS[args.arch]
    dev = "cuda" if torch.cuda.is_available() else "cpu"   # RNG only: none of our kernels
    model = SyntheticLlama(arch, seed=0, alpha=args.alpha, damp_from=args.exit_layer, device=dev)
    sd = model.state_dict(dtype=torch.bfloat16, device="cpu")
    prompts = synthetic_prompts(arch.vocab, 8, args.prompt_len)
    # bounded sample: same prompt length, a short continuation (CPU runs ~0.1-0.6 s per round)
    cores = cpu_threads()
    w, w_dtype = cpu_weights(sd, arch)
    del sd
    # bounded sample of the SAME workload (same architecture, weights, prompts, exit layer, draft
    # count, greedy): the 512-token continuation is cut to 16..64 tokens so that the whole
    # --steps K run stays within --cpu-budget seconds of CPU time
    steps = max(1, args.steps)
    try:
        with time_limit(args.cpu_budget + 240):
            cpu_steps, _spent, prefill_s, round_s = cpu_sized_sample(args, w, arch, prompts, args.cpu_budget / steps)
            if args.cpu_max_steps:
                cpu_steps = args.cpu_max_steps
            tokens, seconds, acc = cpu_reference_run(args, w, arch, prompts, steps, cpu_steps)
    except TimeoutError as exc:
        emit(json.dumps({"impl": "reference", "unavailable": f"CPU run did not finish: {exc}"}))
        return
    value = tokens / seconds
    full = args.max_steps / (prefill_s + args.max_steps * round_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": seconds / steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": f"{w_dtype} (CPU oracle port; the engine arm computes in bf16)",
        "data": "synthetic",
        "config": {"workload": workload_string(args),
                   "sample": f"each step = one generation cut to a {cpu_steps}-token continuation "
                             f"(prefill of {args.prompt_len} ids included); measured prefill {prefill_s:.2f} s, "
                             f"{round_s * 1e3:.0f} ms per round -> {full:.2f} tokens/s extrapolated to the full "
                             f"{args.max_steps}-token continuation"},
        "acceptance_rate": acc,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "cpu": cpu_model_name(),
                         "sample": f"{steps} generations x {cpu_steps} tokens, "
                                   f"prompt {args.prompt_len}, oracle port in torch {w_dtype} on {cores} threads",
                         "prefill_s": prefill_s, "s_per_round": round_s,
                         "extrapolated_full_length_tokens_per_s": full},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
class Watchdog:
    """A hung collective must not cost the driver its JSON line: at the deadline rank 0 prints the
    best line it has (the headline if it finished, else an error line) and EVERY rank exits 0."""

    def __init__(self, seconds: float, rank: int):
        import threading
        self.rank = rank
        self.line = None
        self.note = "started"
        self._t = threading.Timer(seconds, self._fire)
        self._t.daemon = True
        self._t.start()

    def _fire(self):
        if self.rank == 0:
            line = self.line or {"metric": METRIC, "value": None, "unit": UNIT,
                                 "error": f"bench.py watchdog fired during: {self.note}"}
            line.setdefault("extra", {})["watchdog"] = f"deadline hit during: {self.note}"
            emit(json.dumps(line))
        os._exit(0)

    def cancel(self):
        self._t.cancel()


def measure_generations(strat, eng, model, prompts, gcfg, args, eos, first, count, e2e=False):
    """`count` generations starting at prompt index `first`, device-timed: CUDA events on the
    engine's stream around prefill and every round, inputs already resident."""
    out = dict(tokens=0, dev_ms=0.0, bytes=0.0, accs=[], streams=[], last_rounds=[])
    for i in range(count):
        prompt = prompts[(first + i) % len(prompts)]
        eng.begin(exit_layer=gcfg.exit_layer, max_steps=gcfg.max_steps, eos_token_ids=eos)
        eng.prefill(prompt)
        ms = eng.last_device_ms
        toks, matches, drafted, rounds = [], 0, 0, []
        while len(toks) < gcfg.max_steps:
            d = min(gcfg.num_speculations, gcfg.max_steps - len(toks) - 1)
            ctx = eng.kv_len
            r = eng.round(d)
            ms += eng.last_device_ms
            out["bytes"] += eng.round_bytes(d, ctx)
            rounds.append(r)
            toks += r.emitted
            matches += r.n_matches
            drafted += r.n_drafted
            if eos[0] in toks:
                toks = toks[: toks.index(eos[0])]
                break
        out["tokens"] += len(toks)
        out["dev_ms"] += ms
        out["accs"].append(matches / max(1, drafted))
        out["streams"].append(toks)
        out["last_rounds"] = rounds
    return out


def dump_outputs(out_dir, meas):
    """What the timed path handed its caller in the last timed generation, as float64 .npy
    (token ids are exact below 2^53): the generated tokens, the generation's acceptance rate and
    every round's lsk_round_out fields; ragged per-round id lists are concatenated in round order."""
    import numpy as np
    rounds = meas["last_rounds"]
    arrays = {
        "tokens": meas["streams"][-1],
        "acceptance_rate": [meas["accs"][-1]],
        "round_n_drafted": [r.n_drafted for r in rounds],
        "round_n_matches": [r.n_matches for r in rounds],
        "round_kv_len": [r.kv_len for r in rounds],
        "round_draft_ids": [t for r in rounds for t in r.draft],
        "round_verified_ids": [t for r in rounds for t in r.verified],
        "round_emitted_ids": [t for r in rounds for t in r.emitted],
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, values in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(values, dtype=np.float64))


def class_profile(eng, arch, tp, prompts, gcfg, eos, reps=5):
    """Eager rounds with a CUDA-event pair around every launch -> per kernel class time / launches."""
    eng.begin(exit_layer=gcfg.exit_layer, max_steps=gcfg.max_steps, eos_token_ids=eos)
    eng.prefill(prompts[0])
    for _ in range(2):
        eng.round(gcfg.num_speculations)
    cls_ms = {k: 0.0 for k in eng.KERNEL_CLASSES}
    cls_n = {k: 0 for k in eng.KERNEL_CLASSES}
    for _ in range(reps):
        _r, ms, cnt, _tot = eng.profile_round(gcfg.num_speculations)
        for k in ms:
            cls_ms[k] += ms[k]
            cls_n[k] += cnt[k]
    a, t = arch, max(1, tp)
    wb = {"qkv": 2.0 * (a.q_dim + 2 * a.kv_dim) * a.hidden / t, "o_proj": 2.0 * a.hidden * a.q_dim / t,
          "gate_up": 2.0 * 2 * a.inter * a.hidden / t, "down": 2.0 * a.hidden * a.inter / t,
          "lm_head": 2.0 * a.vocab * a.hidden / t}
    return cls_ms, cls_n, wb, reps


def ncu_traffic(arch_name, tp, cls):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r2_ncu_traffic.json, written by tools/ncu_traffic.py from the raw CSV export)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")) as f:
            tab = json.load(f)
        ent = tab.get(f"{arch_name}/tp{tp}", {}).get(cls)
        return float(ent["dram_bytes_per_launch"]) if ent else None
    except Exception:
        return None


def roofline_block(args, arch, tp, eng, prompts, gcfg, eos, meas, peak, peak_kind):
    cls_ms, cls_n, wb, reps = class_profile(eng, arch, tp, prompts, gcfg, eos)
    gemm_bytes = sum(wb[k] * cls_n[k] for k in wb)
    gemm_ms = sum(cls_ms[k] for k in wb)
    gemm_launches = sum(cls_n[k] for k in wb)
    # dominant kernel = the instantiation with the largest share of device time (gate/up projection)
    dom = max(wb, key=lambda k: cls_ms[k])
    dom_us = cls_ms[dom] * 1e3 / max(1, cls_n[dom])
    achieved = wb[dom] / (dom_us * 1e-6) / 1e9
    whole = meas["bytes"] / (meas["dev_ms"] * 1e-3) / 1e9
    return {"bound": "hbm",
            "kernel": f"lsk::gemm_skinny_kernel<1,PRO_RMS/BF16,EPI_*> [{dom}] — TMA-ring weight-streaming GEMM",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
            "bytes_per_launch": wb[dom], "avg_launch_us": dom_us,
            "traffic": ncu_traffic(args.arch, tp, dom),
            "how": "algorithmic bytes (packed weight bytes of the GEMM) / mean CUDA-event duration of "
                   "its launches in eager rounds on the engine stream (includes launch gaps that graph "
                   "replay + PDL hide); traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch "
                   "from the ncu capture under profiles/ (null when no capture of this config is committed)",
            "all_gemm_launches": {"achieved": gemm_bytes / (gemm_ms * 1e-3) / 1e9,
                                  "frac": gemm_bytes / (gemm_ms * 1e-3) / 1e9 / peak,
                                  "launches_per_round": gemm_launches / reps},
            "per_class": {k: {"launches_per_round": cls_n[k] / reps, "ms_per_round": cls_ms[k] / reps,
                              "gbs": (wb[k] * cls_n[k] / (cls_ms[k] * 1e-3) / 1e9) if k in wb and cls_ms[k] > 0 else None}
                          for k in eng.KERNEL_CLASSES},
            "whole_path": {"achieved": whole, "frac": whole / peak,
                           "note": "algorithmic bytes of every round per GPU (weights + KV, SURVEY.md 8(d)) / "
                                   "device time of the timed region (graph replay)"}}


def tp_logits_check(model, arch, prompt, eos, max_ctx, rank, world):
    """max |logit(TP engine) - logit(single-GPU engine)| over the whole vocabulary at the first
    decode step: the sharded engine computes the same function up to fp32 summation order."""
    import torch
    import torch.distributed as dist
    from layerskip_b200.engine import Engine
    vl = arch.vocab // world
    ref = torch.zeros(arch.vocab, dtype=torch.float32, device="cuda")
    if rank == 0:
        e1 = Engine(arch, max_ctx=max_ctx, keep_logits=True)
        e1.load_model(model)
        e1.begin(exit_layer=-1, max_steps=4, eos_token_ids=eos)
        e1.prefill(prompt)
        e1.ar_step()
        ref.copy_(e1.debug_logits(1)[0].cuda())
        e1.close()
    dist.broadcast(ref, src=0)
    et = Engine(arch, max_ctx=max_ctx, keep_logits=True, tp_rank=rank, tp_size=world)
    et.init_comm(None)
    et.load_model(model)
    et.begin(exit_layer=-1, max_steps=4, eos_token_ids=eos)
    et.prefill(prompt)
    et.ar_step()
    mine = et.debug_logits(1)[0].cuda()
    diff = (mine - ref[rank * vl:(rank + 1) * vl]).abs().max().reshape(1)
    scale = ref.abs().max().reshape(1)
    et.close()
    dist.all_reduce(diff, op=dist.ReduceOp.MAX)
    torch.cuda.empty_cache()
    return float(diff.item()), float(scale.item())


def tp_leg(arch_name, exit_layer, args, rank, world, peak, steps=2, warmup=1, single_gpu_check=True):
    """One tensor-parallel measurement over all `world` GPUs: ONE model sharded by heads / FFN
    columns / vocab, one-shot all-reduces over peer-mapped HBM after O-proj and down-proj.  Returns
    tokens/s (device-timed, max over ranks), the per-GPU roofline fraction, and three correctness
    bits: every rank holds the same token stream, speculative == autoregressive on the sharded
    engine, and the stream's agreement with a single-GPU engine of the same model (rank 0)."""
    import torch
    import torch.distributed as dist
    from layerskip_b200 import GenerationConfig
    from layerskip_b200.strategy import (B200AutoRegressiveGenerationStrategy,
                                         B200SelfSpeculativeGenerationStrategy)
    from layerskip_b200.synthetic import synthetic_prompts
    from layerskip_b200.weights import ARCHS, SyntheticLlama
    arch = ARCHS[arch_name]
    if arch.heads % world or arch.kv_heads % world:
        return {"skipped": f"{arch.kv_heads} kv heads do not divide by {world} ranks"}
    model = SyntheticLlama(arch, seed=0, alpha=args.alpha, damp_from=exit_layer, device="cuda")
    max_ctx = ((args.prompt_len + args.max_steps + 64 + 63) // 64) * 64
    prompts = synthetic_prompts(arch.vocab, 8, args.prompt_len)
    eos = [arch.vocab - 1]
    gcfg = GenerationConfig(max_steps=args.max_steps, exit_layer=exit_layer,
                            num_speculations=args.num_speculations, sample=False,
                            generation_strategy="self_speculative")
    short = GenerationConfig(max_steps=48, exit_layer=exit_layer, num_speculations=args.num_speculations,
                             sample=False, generation_strategy="self_speculative")
    single = None
    logit_diff = None
    if single_gpu_check:
        if rank == 0:
            s1 = B200SelfSpeculativeGenerationStrategy(max_ctx=max_ctx)
            single = s1.generate_token_ids(model, prompts[0], eos, short).predicted_tokens
            s1.engines.close()
        dist.barrier()
        logit_diff = tp_logits_check(model, arch, prompts[0], eos, max_ctx, rank, world)
    dist.barrier()
    strat = B200SelfSpeculativeGenerationStrategy(max_ctx=max_ctx, tp_rank=rank, tp_size=world)
    eng = strat.engine_for(model)
    ar = B200AutoRegressiveGenerationStrategy(engine_cache=strat.engines)
    spec_tokens = strat.generate_token_ids(model, prompts[0], eos, short).predicted_tokens
    ar_tokens = ar.generate_token_ids(model, prompts[0], eos,
                                      GenerationConfig(max_steps=48, exit_layer=-1, num_speculations=-1,
                                                       sample=False)).predicted_tokens
    for i in range(warmup):
        measure_generations(strat, eng, model, prompts, gcfg, args, eos, i, 1, e2e=False)
    torch.cuda.synchronize()
    dist.barrier()
    m = measure_generations(strat, eng, model, prompts, gcfg, args, eos, warmup, steps, e2e=False)
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([m["dev_ms"]], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s = float(t.item()) * 1e-3
    # every rank must hold the same stream: compare a hash of all timed tokens
    h = 1469598103934665603
    for tok in [x for st in m["streams"] for x in st] + spec_tokens:
        h = ((h ^ (tok + 1)) * 1099511628211) & 0x7FFFFFFFFFFFFFFF
    hv = torch.tensor([h], dtype=torch.int64, device="cuda")
    lo, hi = hv.clone(), hv.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    cls_ms, cls_n, wb, reps = class_profile(eng, arch, world, prompts, gcfg, eos, reps=3)
    whole = m["bytes"] / (m["dev_ms"] * 1e-3) / 1e9
    res = {"arch": arch_name, "tp": world, "exit_layer": exit_layer,
           "tokens_per_s": m["tokens"] / dev_s, "ms_per_generation": dev_s * 1e3 / steps,
           "generations": steps, "acceptance_rate": sum(m["accs"]) / max(1, len(m["accs"])),
           "per_gpu_hbm_gbs": whole, "per_gpu_roofline_frac": whole / peak,
           "collectives": tp_collectives_name(),
           "per_class": {k: {"launches_per_round": cls_n[k] / reps, "ms_per_round": cls_ms[k] / reps}
                         for k in eng.KERNEL_CLASSES},
           "ranks_agree": bool(int(lo.item()) == int(hi.item())),
           "spec_equals_ar_on_tp_engine": spec_tokens == ar_tokens}
    if logit_diff is not None:
        res["first_step_logits_vs_single_gpu"] = {"max_abs_diff": logit_diff[0], "max_abs_logit": logit_diff[1]}
    if single is not None:
        n_same = 0
        for x, y in zip(single, spec_tokens):
            if x != y:
                break
            n_same += 1
        # informative: fp32 summation order differs between 1 and N ranks, so a near-tie arg-max of
        # a random-init model may flip; the logits check above is the numeric criterion
        res["single_gpu_token_prefix_match"] = f"{n_same}/{len(single)}"
    strat.engines.close()
    del model
    torch.cuda.empty_cache()
    dist.barrier()
    return res


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from layerskip_b200 import GenerationConfig
    from layerskip_b200.strategy import B200SelfSpeculativeGenerationStrategy
    from layerskip_b200.synthetic import synthetic_prompts
    from layerskip_b200.weights import ARCHS, SyntheticLlama

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (use --impl reference for the CPU arm)")
    dog = Watchdog(args.deadline, rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    # N > 1: the headline is ONE model tensor-parallel over the N GPUs (strong scaling, the split
    # north_star names); independent replicas (weak scaling) are reported in extra.replicas
    tp = world if (world > 1 and not args.replicas) else 1

    arch = ARCHS[args.arch]
    if tp > 1 and (arch.heads % tp or arch.kv_heads % tp):
        raise SystemExit(f"{args.arch}: {arch.kv_heads} kv heads do not divide by {tp} ranks")
    model = SyntheticLlama(arch, seed=0, alpha=args.alpha, damp_from=args.exit_layer, device="cuda")
    # KV pool: the workload's context, and room for the 1024-id prefill measurement of the extras
    max_ctx = max(((args.prompt_len + args.max_steps + 64 + 63) // 64) * 64, 1152)
    eos = [arch.vocab - 1]
    gcfg = GenerationConfig(max_steps=args.max_steps, exit_layer=args.exit_layer,
                            num_speculations=args.num_speculations, sample=False,
                            generation_strategy="self_speculative")
    prompts = synthetic_prompts(arch.vocab, 8 * max(1, world), args.prompt_len)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return float(t.item())

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- correctness reference for the TP headline: the single-GPU engine's tokens (rank 0)
    single_tokens = None
    logit_diff = None
    short = GenerationConfig(max_steps=48, exit_layer=args.exit_layer, num_speculations=args.num_speculations,
                             sample=False, generation_strategy="self_speculative")
    if tp > 1:
        dog.note = "single-GPU reference tokens / logits"
        if rank == 0:
            s1 = B200SelfSpeculativeGenerationStrategy(max_ctx=max_ctx)
            single_tokens = s1.generate_token_ids(model, prompts[0], eos, short).predicted_tokens
            s1.engines.close()
        barrier()
        logit_diff = tp_logits_check(model, arch, prompts[0], eos, max_ctx, rank, world)
        barrier()

    dog.note = "engine creation / weight upload"
    strat = B200SelfSpeculativeGenerationStrategy(
        max_ctx=max_ctx, tp_rank=rank if tp > 1 else 0, tp_size=tp)
    eng = strat.engine_for(model)
    my_prompts = prompts if tp > 1 else prompts[rank::world]   # replicas: disjoint prompt streams per GPU

    dog.note = "warm-up"
    for i in range(args.warmup):
        measure_generations(strat, eng, model, my_prompts, gcfg, args, eos, i, 1, e2e=False)
    barrier()
    launches0 = eng.launch_count
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dog.note = "timed region"
    meas = measure_generations(strat, eng, model, my_prompts, gcfg, args, eos, args.warmup, args.steps, e2e=False)
    barrier()
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, meas)
    # e2e leg through the plug-in call (wall clock, host ids in / host ids out, every copy and the
    # per-round sync inside the region)
    e2e = dict(tokens_e2e=0, wall=0.0, rounds=0)
    for i in range(args.steps):
        prompt = my_prompts[(args.warmup + i) % len(my_prompts)]
        w0 = time.perf_counter()
        res = strat.generate_token_ids(model, prompt, eos, gcfg)
        e2e["wall"] += time.perf_counter() - w0
        e2e["tokens_e2e"] += len(res.predicted_tokens)
        e2e["rounds"] += len(strat.last_rounds)
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    t_dev = allmax(meas["dev_ms"]) * 1e-3
    t_wall = allmax(e2e["wall"])
    if tp > 1:        # every rank holds the same stream of tokens
        tokens_total, tokens_total_e2e = meas["tokens"], e2e["tokens_e2e"]
    else:
        tokens_total, tokens_total_e2e = allsum(meas["tokens"]), allsum(e2e["tokens_e2e"])
    value = tokens_total / t_dev
    e2e_value = tokens_total_e2e / t_wall
    peak, peak_kind = measured_peaks()

    tp_check = None
    if tp > 1:
        dog.note = "TP correctness bits"
        from layerskip_b200.strategy import B200AutoRegressiveGenerationStrategy
        spec_tokens = strat.generate_token_ids(model, prompts[0], eos, short).predicted_tokens
        ar_tokens = B200AutoRegressiveGenerationStrategy(engine_cache=strat.engines).generate_token_ids(
            model, prompts[0], eos, GenerationConfig(max_steps=48, exit_layer=-1, num_speculations=-1,
                                                     sample=False)).predicted_tokens
        h = 1469598103934665603
        for tok in [x for st in meas["streams"] for x in st] + spec_tokens:
            h = ((h ^ (tok + 1)) * 1099511628211) & 0x7FFFFFFFFFFFFFFF
        hv = torch.tensor([h], dtype=torch.int64, device="cuda")
        lo, hi = hv.clone(), hv.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        tp_check = {"ranks_agree": bool(int(lo.item()) == int(hi.item())),
                    "spec_equals_ar_on_tp_engine": spec_tokens == ar_tokens}
        if single_tokens is not None:
            n_same = 0
            for x, y in zip(single_tokens, spec_tokens):
                if x != y:
                    break
                n_same += 1
            tp_check["single_gpu_token_prefix_match"] = f"{n_same}/{len(single_tokens)}"
        if logit_diff is not None:
            tp_check["first_step_logits_vs_single_gpu"] = {"max_abs_diff": logit_diff[0],
                                                           "max_abs_logit": logit_diff[1]}

    # ---- roofline of the dominant kernel (weight-streaming skinny GEMM), measured live
    dog.note = "per-class profile"
    roof = None
    if rank == 0 or tp > 1:       # tensor-parallel: every rank must issue the same engine calls
        roof = roofline_block(args, arch, tp, eng, my_prompts, gcfg, eos, meas, peak, peak_kind)

    acc_mean = sum(meas["accs"]) / max(1, len(meas["accs"]))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_dev * 1e3 / max(1, args.steps),
        # the headline series over N is ONE model on N GPUs (tensor parallel): strong scaling, with
        # N = 1 as its first point; `--replicas` makes the independent-replicas series the headline
        "higher_is_better": True, "scaling": "weak" if (args.replicas and world > 1) else "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "acceptance_rate": acc_mean,
        "config": {"workload": workload_string(args),
                   "parallelism": f"tp{tp}" if tp > 1 else ("single-gpu" if world == 1 else f"replicas{world}"),
                   **({"tp_collectives": tp_collectives_name()} if tp > 1 else {}),
                   "l2": "inputs_exceed_l2 (weights 13.5 GB >> 126 MB L2)",
                   "step": "one full generation (prefill + rounds)"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * args.prompt_len,
                "d2h_bytes_per_step": int(e2e["rounds"] / max(1, args.steps)) * 212},
        "gpu_launches": int(launches),
        "roofline": roof, "cpu_baseline": None, "extra": {},
    }
    if tp_check is not None:
        line["tp_check"] = tp_check
    dog.line = line
    extra = line["extra"]

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        dog.note = "cpu baseline"
        try:
            sd = model.state_dict(dtype=torch.bfloat16, device="cpu")
            w, w_dtype = cpu_weights(sd, arch)
            del sd
            cores = cpu_threads()
            t0 = time.perf_counter()
            with time_limit(150):
                n_cpu, _spent, pre_s, rnd_s = cpu_sized_sample(args, w, arch, prompts, 25.0)
                toks, secs, _acc = cpu_reference_run(args, w, arch, prompts, 1, n_cpu)
            line["cpu_baseline"] = {"value": toks / secs, "unit": UNIT, "cores": cores, "kind": "port",
                                    "cpu": cpu_model_name(),
                                    "sample": f"1 generation x {n_cpu} tokens, prompt {args.prompt_len} ids "
                                              f"(prefill included), oracle port in torch {w_dtype} on {cores} threads; "
                                              f"{time.perf_counter() - t0:.1f} s of CPU work incl. sizing probe; "
                                              f"prefill {pre_s:.2f} s + {rnd_s * 1e3:.0f} ms per round"}
            del w
        except Exception as exc:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cpu_threads(), "kind": "port",
                                    "sample": f"failed: {exc!r}"}

    if rank == 0 and not args.no_extra and world == 1:
        dog.note = "extra legs"
        single_gpu_extras(args, arch, strat, eng, model, prompts, eos, extra)

    strat.engines.close()
    del model
    torch.cuda.empty_cache()

    if world > 1 and not args.no_extra:
        # ---- the other parallel legs of BASELINE.json's configs on the same N GPUs
        legs = {}
        try:
            if tp > 1:
                dog.note = "replicas leg"
                legs_rep = replicas_leg(args, rank, world, local_rank)
                if rank == 0:
                    extra["replicas"] = legs_rep
            dog.note = "13B tensor-parallel leg"
            legs["llama2-13b"] = tp_leg("llama2-13b", 8, args, rank, world, peak)
            if world == 8:
                dog.note = "70B tensor-parallel leg"
                legs["llama2-70b"] = tp_leg("llama2-70b", 10, args, rank, world, peak, single_gpu_check=False)
        except Exception as exc:  # pragma: no cover
            legs["error"] = repr(exc)
        if rank == 0:
            extra["tp"] = legs

    if rank == 0:
        dog.cancel()
        emit(json.dumps(line))
    else:
        dog.cancel()
    if world > 1:
        dist.destroy_process_group()


def replicas_leg(args, rank, world, local_rank):
    """N independent single-GPU engines serving disjoint prompt streams (weak scaling, no
    data-path collective): aggregate tokens/s = all tokens / max-over-ranks device time."""
    import torch
    import torch.distributed as dist
    from layerskip_b200 import GenerationConfig
    from layerskip_b200.strategy import B200SelfSpeculativeGenerationStrategy
    from layerskip_b200.synthetic import synthetic_prompts
    from layerskip_b200.weights import ARCHS, SyntheticLlama
    arch = ARCHS[args.arch]
    model = SyntheticLlama(arch, seed=0, alpha=args.alpha, damp_from=args.exit_layer, device="cuda")
    max_ctx = ((args.prompt_len + args.max_steps + 64 + 63) // 64) * 64
    strat = B200SelfSpeculativeGenerationStrategy(max_ctx=max_ctx)
    eng = strat.engine_for(model)
    prompts = synthetic_prompts(arch.vocab, 8 * world, args.prompt_len)[rank::world]
    eos = [arch.vocab - 1]
    gcfg = GenerationConfig(max_steps=args.max_steps, exit_layer=args.exit_layer,
                            num_speculations=args.num_speculations, sample=False,
                            generation_strategy="self_speculative")
    measure_generations(strat, eng, model, prompts, gcfg, args, eos, 0, 1, e2e=False)
    torch.cuda.synchronize()
    dist.barrier()
    m = measure_generations(strat, eng, model, prompts, gcfg, args, eos, 1, 2, e2e=False)
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([m["dev_ms"]], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    n = torch.tensor([float(m["tokens"])], dtype=torch.float64, device="cuda")
    dist.all_reduce(n)
    strat.engines.close()
    del model
    torch.cuda.empty_cache()
    dist.barrier()
    return {"parallelism": f"replicas{world}", "scaling": "weak", "generations_per_rank": 2,
            "tokens_per_s": float(n.item()) / (float(t.item()) * 1e-3),
            "note": "independent 7B engines, disjoint prompt streams, no data-path collective"}


def single_gpu_extras(args, arch, strat, eng, model, prompts, eos, extra):
    """Informative single-GPU legs: autoregressive on the same engine, acceptance-controlled
    models, the reference's default sampling mode."""
    import torch
    from layerskip_b200.weights import SyntheticLlama
    try:
        eng.begin(exit_layer=-1, max_steps=args.max_steps, eos_token_ids=eos)
        eng.prefill(prompts[0])
        ms, nb = eng.last_device_ms, 0.0
        for _ in range(128):
            ctx = eng.kv_len
            eng.ar_step()
            ms += eng.last_device_ms
            nb += eng.ar_bytes(ctx)
        extra["autoregressive_same_engine"] = {"tokens_per_s": 128 / (ms * 1e-3),
                                               "hbm_gbs": nb / (ms * 1e-3) / 1e9}
    except Exception as exc:  # pragma: no cover
        extra["autoregressive_same_engine"] = {"error": repr(exc)}
    # prefill alone (tcgen05 GEMM path): device time of lsk_prefill for 128 and 1024 prompt ids
    try:
        pf = {}
        for n in (128, 1024):
            if n + 8 > eng.max_ctx:
                continue
            ids = (prompts[0] * (n // len(prompts[0]) + 1))[:n]
            eng.begin(exit_layer=args.exit_layer, max_steps=4, eos_token_ids=eos)
            eng.prefill(ids)
            eng.begin(exit_layer=args.exit_layer, max_steps=4, eos_token_ids=eos)
            eng.prefill(ids)
            pf[str(n)] = {"ms": eng.last_device_ms}
        extra["prefill_ms"] = pf
    except Exception as exc:  # pragma: no cover
        extra["prefill_ms"] = {"error": repr(exc)}
    # acceptance-controlled legs (SURVEY.md App. C): o_proj/down_proj of layers >= E damped by
    # alpha; same architecture, prompts and settings, one 512-token generation each
    sweep = []
    for alpha in ([] if args.alpha != 1.0 else [0.3, 0.1, 0.03]):
        try:
            strat.engines.close()
            m2 = SyntheticLlama(arch, seed=0, alpha=alpha, damp_from=args.exit_layer, device="cuda")
            e2 = strat.engine_for(m2)
            tot_ms, n_tok, mt, dr = 0.0, 0, 0, 0
            for rep in range(2):        # rep 0 warms the graphs up
                e2.begin(exit_layer=args.exit_layer, max_steps=args.max_steps, eos_token_ids=eos)
                e2.prefill(prompts[1])
                ms = e2.last_device_ms
                out = []
                while len(out) < args.max_steps:
                    r = e2.round(min(args.num_speculations, args.max_steps - len(out) - 1))
                    ms += e2.last_device_ms
                    out += r.emitted
                    if rep == 1:
                        mt += r.n_matches
                        dr += r.n_drafted
                if rep == 1:
                    tot_ms, n_tok = ms, len(out)
            sweep.append({"alpha": alpha, "acceptance_rate": mt / max(1, dr),
                          "tokens_per_s": n_tok / (tot_ms * 1e-3)})
            del m2
        except Exception as exc:  # pragma: no cover
            sweep.append({"alpha": alpha, "error": repr(exc)})
    if sweep:
        extra["acceptance_sweep"] = sweep
    # the reference's DEFAULT decoding mode (sample=True, T=0.6, top_p=0.9; generator_base.py:39-42)
    try:
        strat.engines.close()
        eng_s = strat.engine_for(model)
        tot_ms, n_tok, mt, dr = 0.0, 0, 0, 0
        for rep in range(2):
            eng_s.begin(exit_layer=args.exit_layer, max_steps=args.max_steps, eos_token_ids=eos,
                        sample=True, temperature=0.6, top_k=0, top_p=0.9, seed=1234 + rep)
            eng_s.prefill(prompts[2 % len(prompts)])
            ms = eng_s.last_device_ms
            out = []
            while len(out) < args.max_steps:
                r = eng_s.round(min(args.num_speculations, args.max_steps - len(out) - 1))
                ms += eng_s.last_device_ms
                out += r.emitted
                if rep == 1:
                    mt += r.n_matches
                    dr += r.n_drafted
            if rep == 1:
                tot_ms, n_tok = ms, len(out)
        extra["sampling_T0.6_top_p0.9"] = {"acceptance_rate": mt / max(1, dr),
                                           "tokens_per_s": n_tok / (tot_ms * 1e-3)}
    except Exception as exc:  # pragma: no cover
        extra["sampling_T0.6_top_p0.9"] = {"error": repr(exc)}


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The ONE JSON line goes to the process's original stdout; everything else any library
    prints to fd 1 (NCCL's version banner, for one) was rerouted to stderr in main()."""
    data = (line + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line + "\n")
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
