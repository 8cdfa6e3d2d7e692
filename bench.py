#!/usr/bin/env python
"""bench.py — decode tokens/s of the sync speculative-decoding hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu]
                    [--workload 70b|8b|qwen32b|tiny] [--temp T] [--lm-scale S] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: K_spec+1 draft forwards -> one (K_spec+1)-token target
forward -> accept/reject+resample.  Workload (N=1 default): Llama-3.1-70B target + Llama-3.2-1B draft, k=6, b=1,
temp 0, synthetic "bigram agreement" weights at the exact shapes (there are no checkpoints in the image), random
128-token prompt.  Prints ONE JSON line (rank 0):

  value     decode tokens/s, device-resident loop (inputs already in HBM; CUDA events; max over ranks)
  e2e       the same metric through the public engine API (LLMEngine.step: scheduler + ssdk_spec_step with HOST
            buffers: per-step H2D of ctx/recovery/block tables and D2H of tokens/accept count inside the timing)
  roofline  achieved HBM GB/s of the dominant kernel (weight-streaming tcgen05 GEMM, largest instance) vs the
            measured peak, plus the whole-step fraction of the HBM roofline of SURVEY §8(d)
  cpu_baseline  the oracle (CPU restatement of the reference path) timed on the host cores on a bounded sample
  parity_check  temp 0: the tokens of the timed device-resident loop AND of the engine (e2e) loop against the closed-form
            greedy chain of the synthetic target (t_{i+1} = pi_t(t_i)) — token-for-token, at every N
  allreduce "symm" (one-shot NVLink all-reduce, ssd_b200's own kernels) | "nccl" (SSD_B200_NO_SYMM=1) | "none" (N=1)
  reference_gpu  (N=1) the UNMODIFIED reference engine on this box's GPU (baseline/ref_gpu.py: torch.compile, cuBLAS,
            its CUDA graphs, flash_attn 2.8.3 stub) on the same weights and prompt: its tokens/s, and whether its tokens
            equal ours; `--impl reference-gpu` prints that arm alone
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "70b": ("llama-3.1-70b", "llama-3.2-1b", "Llama-3.1-70B target + Llama-3.2-1B draft"),
    "8b": ("llama-3.1-8b", "llama-3.2-1b", "Llama-3.1-8B target + Llama-3.2-1B draft"),
    "qwen32b": ("qwen3-32b", "qwen3-0.6b", "Qwen3-32B target + Qwen3-0.6B draft"),
    "tiny": ("llama-tiny-target", "llama-tiny-draft", "tiny Llama pair (plumbing)"),
}
# forward weight bytes (bf16, body + lm_head) and KV bytes/token: SURVEY §2 / BASELINE.md §3
W_BYTES = {"llama-3.2-1b": 2.472e9, "llama-3.1-8b": 15.010e9, "llama-3.1-70b": 139.006e9, "qwen3-0.6b": 1.192e9,
           "qwen3-32b": 63.968e9}
KV_BYTES = {"llama-3.2-1b": 32768, "llama-3.1-8b": 131072, "llama-3.1-70b": 327680, "qwen3-0.6b": 114688,
            "qwen3-32b": 262144}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while a timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int = 0):
        self.gpu, self.rows, self._stop, self._t = gpu, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max([int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(self.rows)}


def usable_cores() -> int:
    """Threads the CPU arm may really use: min(CPU affinity, cgroup cpu.max quota).  os.cpu_count() reports the host's
    128 logical CPUs while the container's quota is 16 — 128 oversubscribed threads made the round-1 CPU arm swing 13x."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def run_reference_gpu_subprocess(args, timeout_s: int = 480):
    """bench.py --impl reference-gpu / the `reference_gpu` object of the default line: baseline/ref_gpu.py in its own
    process (the reference calls os._exit from an atexit hook, and both engines cannot hold a 70B model at once)."""
    out_path = os.path.join(tempfile.mkdtemp(prefix="ssd_refgpu_"), "ref.json")
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_gpu.py"), "--workload", args.workload, "--steps", str(args.steps),
           "--warmup", str(args.warmup), "--spec-k", str(args.spec_k), "--alpha", str(args.alpha), "--prompt-len",
           str(args.prompt_len), "--temp", str(args.temp), "--out", out_path]
    if args.lm_scale:
        cmd += ["--lm-scale", str(args.lm_scale)]
    t0 = time.time()
    res = None
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
        with open(out_path) as f:
            d = json.loads(f.read())
    except Exception as exc:  # noqa: BLE001  (timeout, crash before the result file was written, malformed result)
        tail = (res.stdout + res.stderr)[-300:] if res is not None else ""
        d = {"impl": "reference-gpu", "unavailable": f"{type(exc).__name__}: {exc} {tail}"[:500]}
    finally:
        shutil.rmtree(os.path.dirname(out_path), ignore_errors=True)
    d["wall_s"] = round(time.time() - t0, 1)
    return d


def bytes_per_step(tshape, dshape, K, ctx, tp):
    """SURVEY §8(d): (K+1)(W_draft + ctx*kv_d) + (W_target + ctx*kv_t)/TP + (2K+1)*V*2."""
    V = 151936 if "qwen" in tshape else 128256
    if tshape not in W_BYTES:
        return None
    return (K + 1) * (W_BYTES[dshape] + ctx * KV_BYTES[dshape]) + (W_BYTES[tshape] + ctx * KV_BYTES[tshape]) / tp + (2 * K + 1) * V * 2


# ----------------------------------------------------------------------------------------------- ours
def run_ours(args):
    import torch
    import torch.distributed as dist

    from ssd_b200 import synth
    from ssd_b200.engine import llm_engine
    from ssd_b200.llm import LLM
    from ssd_b200.sampling_params import SamplingParams

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    tshape, dshape, desc = WORKLOADS[args.workload]
    K = args.spec_k
    root = tempfile.mkdtemp(prefix="ssd_b200_bench_")
    need = args.prompt_len + (args.steps + max(args.warmup, 3) + 6) * (K + 1) + 64
    max_len = max(4096, -(-need // 256) * 256)
    ref_gpu = None
    if world == 1 and not args.no_ref_gpu and args.workload != "tiny":
        ref_gpu = run_reference_gpu_subprocess(args)  # BEFORE our engine takes the GPU memory (70B: 141 GB each)
    tdir = synth.make_model_dir(root, tshape, "target", seed=0, alpha=args.alpha, lm_scale=args.lm_scale)
    ddir = synth.make_model_dir(root, dshape, "draft", seed=0, alpha=args.alpha, lm_scale=args.lm_scale)
    temp = float(args.temp)
    t_init = time.time()
    llm = LLM(tdir, speculate=True, draft=ddir, speculate_k=K, num_gpus=world, max_num_seqs=1, max_model_len=max_len,
              kvcache_block_size=256, jit_speculate=True, enforce_eager=False, use_pdl=not args.no_pdl, verbose=False)
    init_s = time.time() - t_init
    runner = llm.runner
    import random
    random.seed(0)
    prompt = [random.randint(0, 10000) % synth.SHAPES[tshape][6] for _ in range(args.prompt_len)]
    steps, warm = args.steps, args.warmup
    budget_tokens = (steps + warm + 4) * (K + 1) + 8

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- kernel-only: device-resident loop ----------------
    from ssd_b200 import lib as L
    nblk = runner.max_blocks
    bt = list(range(nblk))
    rec = runner.prefill(L.TARGET, prompt, bt)
    runner.prefill(L.DRAFT, prompt, bt, want_sample=False)
    runner.stage([len(prompt)], [rec], [bt], [bt], [temp], [temp])
    for _ in range(warm):
        runner.step_resident(1)
    sync_all()
    _, tot0, _ = runner.fetch(1)
    l0 = runner.launch_count
    with ClockSampler(local) as cs:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for _ in range(steps):
            runner.step_resident(1)
        e1.record()
        sync_all()
    ms_dev = e0.elapsed_time(e1)
    last_spec, tot1, last_rec = runner.fetch(1)
    dev_log = runner.resident_log(0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, runner, last_spec, tot1, last_rec, dev_log)
    launches = runner.launch_count - l0
    toks_dev = int(tot1[0] - tot0[0])
    if world > 1:
        t = torch.tensor([ms_dev], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev = float(t[0])
    clocks = cs.summary()
    ctx_mid = len(prompt) + (tot0[0] + tot1[0]) // 2

    # ---------------- end to end: public engine API, host buffers every step ----------------
    e2e = None
    if rank == 0 or world > 1:
        llm.add_request(prompt, SamplingParams(temperature=temp, max_new_tokens=budget_tokens, ignore_eos=True))
        e2e_seq = llm.scheduler.waiting[-1]
        step = llm.create_inference_step(llm.config)
        for k in llm_engine.METRICS:
            llm_engine.METRICS[k] = [] if isinstance(llm_engine.METRICS[k], list) else 0
        llm.step(step)  # prefill
        for _ in range(warm):
            llm.step(step)
        sync_all()
        tok0 = llm_engine.METRICS["decode_total_tokens"]
        t0 = time.perf_counter()
        for _ in range(steps):
            llm.step(step)
        sync_all()
        dt = time.perf_counter() - t0
        toks = llm_engine.METRICS["decode_total_tokens"] - tok0
        lens = llm_engine.METRICS["accepted_suffix_lens_with_recovery"]
        e2e = {"value": toks / dt, "unit": "tokens/s", "h2d_bytes_per_step": int(runner.step_io_bytes()[0]),
               "d2h_bytes_per_step": int(runner.step_io_bytes()[1]), "ms_per_step": dt / steps * 1e3,
               "accept_len": sum(lens) / max(1, len(lens))}
        e2e_tokens = list(e2e_seq.completion_token_ids)

    if rank != 0:
        if world > 1:
            try:
                dist.barrier()
                dist.destroy_process_group()
            except Exception:
                pass
        return
    # ---------------- parity: the generated tokens against the closed-form greedy chain of the synthetic target ----------------
    parity = None
    if temp == 0.0 and not args.lm_scale:
        pi_t, _ = synth.permutations(synth.SHAPES[tshape][6], 0, args.alpha, "cpu")
        pi_t = pi_t.tolist()

        def chain_mismatches(first_prev, toks_):
            bad, prev = 0, first_prev
            for t in toks_:
                bad += int(t != pi_t[prev])
                prev = t
            return bad

        # resident log: first entry = the recovery token sampled by the prefill = pi_t(last prompt token)
        m_dev = chain_mismatches(prompt[-1], dev_log)
        m_e2e = chain_mismatches(prompt[-1], e2e_tokens)
        parity = {"tokens": len(dev_log) + len(e2e_tokens), "mismatches": m_dev + m_e2e,
                  "device_loop": {"tokens": len(dev_log), "mismatches": m_dev},
                  "engine_loop": {"tokens": len(e2e_tokens), "mismatches": m_e2e},
                  "against": "t[i+1] == pi_target(t[i]) from the last prompt token (greedy chain of the synthetic target)"}
        if ref_gpu and ref_gpu.get("tokens"):
            n = min(len(ref_gpu["tokens"]), len(e2e_tokens))
            ref_gpu["tokens_compared_with_ours"] = n
            ref_gpu["token_mismatches_vs_ours"] = sum(int(a != b) for a, b in zip(ref_gpu["tokens"][:n], e2e_tokens[:n]))
        if parity["mismatches"]:
            print(f"[bench] PARITY FAILURE: {parity}", file=sys.stderr, flush=True)
    if ref_gpu is not None:
        ref_gpu.pop("tokens", None)
        if "value" in ref_gpu and e2e:
            ref_gpu["ours_e2e_over_reference_gpu"] = e2e["value"] / ref_gpu["value"]
    # ---------------- roofline ----------------
    peak, peak_src = measured_peaks()
    accept_len = toks_dev / steps
    bstep = bytes_per_step(tshape, dshape, K, int(ctx_mid), world)
    roof = gemm_roofline(runner, peak) if args.workload != "tiny" else None
    step_frac = (bstep / (ms_dev / steps * 1e-3) / 1e9 / peak) if bstep else None
    if roof is not None:
        roof.update({"peak": peak, "peak_source": peak_src, "step_bytes": bstep, "step_frac": step_frac})
    # the CPU baseline is measured on rank 0 at N=1 only (host cores are shared by the ranks otherwise)
    cpu = cpu_baseline(tshape, dshape, K, args.alpha, sample_steps=3) if (not args.no_cpu and world == 1) else None
    out = {
        "metric": "decode tokens/sec (sync speculative decoding, accept-len reported)", "value": toks_dev / (ms_dev * 1e-3),
        "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": ms_dev / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "accept_len": accept_len,
        "config": {"workload": f"{desc}, sync SD k={K} b=1 temp={temp:g}, TP={world}, prompt {args.prompt_len} random tokens, "
                               f"synthetic bigram-agreement weights alpha={args.alpha} (expected accept-len "
                               f"{synth.expected_tokens_per_step(args.alpha, K):.2f})",
                   "l2": "inputs larger than L2: every step streams the full weight set (>= 2.4 GB) through HBM",
                   "init_s": round(init_s, 1)},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
        "parity_check": parity,
        "allreduce": ("none" if world == 1 else ("symm" if getattr(runner, "symm", False) else "nccl")),
        "draft_path": "kernel-per-op" if os.environ.get("SSDK_DRAFT_STREAM", "1") == "0"
        else "draft_stream_kernel (one launch per step; kernel-per-op graph beyond 1024 tokens of context)",
        "reference_gpu": ref_gpu,
    }
    if args.lm_scale:
        out["config"]["lm_scale"] = args.lm_scale
    print(json.dumps(out), flush=True)
    if world > 1:
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass


def dump_outputs(out_dir, runner, spec, total, rec, log):
    """What the timed device-resident loop handed back after its last step, as .npy files (float64 for token ids and
    counts, float32 for logits) so that two builds can be compared output for output on the same seeded inputs:
    that step's speculations [1, K+1], the running count of emitted tokens, the recovery token, every token emitted
    since the prefill, and the target [1, K+1, V] and draft [1, K, V] logits of that step (about 7 MB at V = 128256)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"speculations": spec.astype(np.float64), "tokens_total": total.astype(np.float64),
              "recovery": rec.astype(np.float64), "emitted_tokens": np.asarray(log, dtype=np.float64),
              "logits_target": runner.logits_p(1).float().cpu().numpy(),
              "logits_draft": runner.logits_q(1).float().cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def gemm_roofline(runner, peak):
    """Dominant kernel = gemm_ws_kernel; its largest instance is the target's gate|up projection at M=K+1.
    achieved = algorithmic bytes (weight bytes of that matrix, SURVEY §8d: out*in*2) / CUDA-event time."""
    import torch
    from ssd_b200 import lib as L, ops
    w = runner.weights[L.TARGET]["layers"][0]["gate_up"]
    M = runner.K + 1
    x = torch.randn(M, w.shape[1], device=w.device).to(torch.bfloat16)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=w.device)
    for _ in range(3):
        ops.gate_up_silu(x, w)
    ts = []
    for _ in range(12):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.gate_up_silu(x, w)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = sum(ts) / len(ts)
    nbytes = w.numel() * 2
    ach = nbytes / (ms * 1e-3) / 1e9
    name = f"gemm_ws_kernel<16,EPI_SILU> gate|up [{w.shape[0]}x{w.shape[1]}] M={M}"
    traffic = None  # dram__bytes_read+write of the same launch from the committed ncu --set full capture, if it matches
    try:
        with open(os.path.join(ROOT, "profiles", "gemm_traffic.json")) as f:
            t = json.load(f)
        if t["kernel"] == name:
            traffic = t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:
        pass
    return {"bound": "hbm", "kernel": name, "achieved": ach, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
            "launch_ms": ms, "bytes_per_launch": nbytes}


# ---------------------------------------------------------------------------------------- CPU baseline
def cpu_baseline(tshape, dshape, K, alpha, sample_steps=3, t_layers=2, d_layers=2):
    """The oracle (CPU restatement of the reference's path, torch bf16 on all host cores) on a BOUNDED sample:
    true widths / vocab, but only `t_layers` target and `d_layers` draft decoder layers; the per-layer time is
    extrapolated to the full depth.  Reported baseline, not a target."""
    import torch
    from oracle.model import ModelCfg, OracleModel
    from oracle.spec import SpecSession, contiguous_block_tables
    from ssd_b200 import synth

    def cfg(shape, layers):
        h, L, H, KV, hd, ffn, V, eps, theta, mtype, tied = synth.SHAPES[shape]
        return ModelCfg(hidden=h, layers=layers, heads=H, kv_heads=KV, head_dim=hd, ffn=ffn, vocab=V, rms_eps=eps,
                        rope_theta=theta, qk_norm=(mtype == "qwen3"), max_pos=1024), L

    def weights(c, seed):
        g = torch.Generator().manual_seed(seed)
        mk = lambda r, cc, s: (torch.randn(r, cc, generator=g) * s).to(torch.bfloat16)
        w = {"embed": mk(c.vocab, c.hidden, 1.0), "final_norm": torch.ones(c.hidden, dtype=torch.bfloat16), "layers": []}
        w["lm_head"] = mk(c.vocab, c.hidden, 0.02)
        for _ in range(c.layers):
            lw = {"input_norm": torch.ones(c.hidden, dtype=torch.bfloat16), "post_norm": torch.ones(c.hidden, dtype=torch.bfloat16),
                  "qkv": mk((c.heads + 2 * c.kv_heads) * c.head_dim, c.hidden, 0.02), "o": mk(c.hidden, c.heads * c.head_dim, 0.02),
                  "gate_up": mk(2 * c.ffn, c.hidden, 0.02), "down": mk(c.hidden, c.ffn, 0.02)}
            if c.qk_norm:
                lw["q_norm"] = torch.ones(c.head_dim, dtype=torch.bfloat16)
                lw["k_norm"] = torch.ones(c.head_dim, dtype=torch.bfloat16)
            w["layers"].append(lw)
        return w

    cores = usable_cores()
    torch.set_num_threads(cores)
    tc, tL = cfg(tshape, t_layers)
    dc, dL = cfg(dshape, d_layers)
    t = OracleModel(tc, weights(tc, 1), 2, 256)
    d = OracleModel(dc, weights(dc, 2), 2, 256)
    s = SpecSession(t, d, K, 2)
    bt = contiguous_block_tables(1, 2)
    s.prefill([[5, 6, 7, 8]], [0.0], bt, bt.clone())
    timing = {}

    def timed(tag, fn):
        t0 = time.perf_counter()
        out = fn()
        timing[tag] = timing.get(tag, 0.0) + time.perf_counter() - t0
        return out

    # instrument per-model forward time to separate layer time from embedding / head time
    orig_fwd = SpecSession._forward
    def fwd(self, model, ids, ctx0, q_len, btab):
        return timed("t_fwd" if model is t else "d_fwd", lambda: orig_fwd(self, model, ids, ctx0, q_len, btab))
    SpecSession._forward = fwd
    try:
        s.spec_step()  # warm-up
        timing.clear()
        t0 = time.perf_counter()
        for _ in range(sample_steps):
            s.spec_step()
        wall = (time.perf_counter() - t0) / sample_steps
    finally:
        SpecSession._forward = orig_fwd
    t_fwd, d_fwd = timing["t_fwd"] / sample_steps, timing["d_fwd"] / sample_steps
    other = wall - t_fwd - d_fwd  # lm_head GEMMs + sampler + verify
    full = t_fwd * (tL / t_layers) + d_fwd * (dL / d_layers) + other
    acc = synth.expected_tokens_per_step(alpha, K)
    return {"value": acc / full, "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"{sample_steps} spec steps of the oracle at true widths/vocab with {t_layers}/{tL} target and "
                      f"{d_layers}/{dL} draft layers ({wall:.2f} s/step measured); layer time extrapolated to full depth "
                      f"({full:.1f} s/step) at the synthetic accept-len {acc:.2f}"}


def run_reference(args):
    """Reference arm of this tier: the reference's own CPU implementation of the path = the oracle port
    (the Python reference cannot travel to the GPU box), all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tshape, dshape, desc = WORKLOADS[args.workload]
    K = args.spec_k
    cpu = cpu_baseline(tshape, dshape, K, args.alpha, sample_steps=max(1, min(args.steps, 4)))
    out = {"impl": "reference", "metric": "decode tokens/sec (sync speculative decoding, accept-len reported)",
           "value": cpu["value"], "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
           "data": "synthetic",
           "config": {"workload": f"{desc}, sync SD k={K} b=1 temp=0 — CPU oracle port of the reference path on host cores"},
           "cpu_baseline": cpu,
           "e2e": {"value": cpu["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--temp", type=float, default=0.0, help="sampling temperature of target and draft (BASELINE config 4: 0.7)")
    ap.add_argument("--lm-scale", type=float, default=None, help="synthetic lm_head scale (softens the distribution for temp>0)")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference GPU arm inside the default line")
    ap.add_argument("--workload", default="70b", choices=sorted(WORKLOADS))
    ap.add_argument("--spec-k", type=int, default=6)
    ap.add_argument("--alpha", type=float, default=0.85)
    ap.add_argument("--prompt-len", type=int, default=128)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-gpu":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(run_reference_gpu_subprocess(args)), flush=True)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
