#!/usr/bin/env python
"""bench.py -- decode tokens/s of the crabml CUDA backend on synthetic Llama-2-7B shapes (BASELINE.json metric).

One "step" = one decoded token = one pass of the hot path (225 quantized matvecs + the small ops around them).
  value : device-resident throughput (weights + KV in HBM, no host<->device traffic inside the timed region)
  e2e   : the same loop through the reference-facing runner API with HOST buffers: per step the token id goes
          host->device and the 128 KB logits come device->host (Llama2Runner::forward -> export, llama2.rs:209),
          then the host samples (argmax) and feeds the next token.
  roofline : the dominant kernel (the ffn_gate/ffn_up-shaped matvec, 11008x4096) timed with CUDA events
  cpu_baseline : the CPU restatement of the reference's AVX2 path (oracle/, all host threads) on a bounded sample
`--impl reference` runs ONLY that CPU path and prints the same line shape.
`--dump-outputs DIR` writes what the timed path computed in its last timed step (logits as float32, token ids as float64, a
fixed seeded sample of the prefill GEMM outputs) to DIR/<name>.npy; the inputs are seeded, so two builds run with the same
arguments can be compared output for output.
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
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEED = 0x5EED
WORKLOADS = {
    # name: (config name, body weight type, classifier weight type)
    "llama2-7b-q8_0": ("LLAMA2_7B", "Q8_0", "Q8_0"),
    "llama2-7b-q4_0": ("LLAMA2_7B", "Q4_0", "Q4_0"),
    "llama2-7b-q4_0-q6k": ("LLAMA2_7B", "Q4_0", "Q6_K"),
    "llama2-7b-q4_k": ("LLAMA2_7B", "Q4_K", "Q6_K"),
    "tinyllamas-15m-q8_0": ("TINYLLAMAS_15M", "Q8_0", "Q8_0"),
    # BASELINE.json config 5: the dense matmuls of a 4096-token prefill (TMA + tcgen05 path, csrc/prefill_gemm.cu); see run_prefill
    "mistral-7b-q8_0-prefill": ("MISTRAL_7B", "Q8_0", "Q8_0"),
    "llama2-7b-q8_0-prefill": ("LLAMA2_7B", "Q8_0", "Q8_0"),
}
# dram bytes per megakernel launch from the committed ncu --set full capture (profiles/); None until captured
TRAFFIC = {("llama2-7b-q8_0", 1): 7040893000 + 49879296}     # profiles/r02p_mega_ring_q8_0_ncu_raw.csv (mega_ring_kernel: dram__bytes_read.sum + dram__bytes_write.sum)
MEGA_NAMES = {1: ("mega_kernel", "mega.cu, weights through registers"), 2: ("mega_ring_kernel", "mega_ring.cu, weights through a TMA-fed shared-memory ring")}
TYPE_ID = {"Q4_0": 2, "Q4_1": 3, "Q5_0": 6, "Q5_1": 7, "Q8_0": 8, "Q2_K": 10, "Q3_K": 11, "Q4_K": 12, "Q5_K": 13, "Q6_K": 14}


def usable_cpus():
    """CPUs this process may actually use: affinity mask capped by the cgroup CPU quota (spin-waiting workers beyond the
    quota get throttled by CFS and make the CPU arm erratic)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path restated (oracle/), AVX2 order, all host threads, bounded sample
# --------------------------------------------------------------------------------------------------------------
def cpu_reference_tokens_per_s(workload: str, steps: int = 8, warmup: int = 2, sample_layers: int = 8):
    from crabml_b200 import runner as R          # config table + byte accounting only (no GPU use)
    from oracle import oracle as oc
    from oracle.llama_replay import Llama2Runner, LlamaConfig, LlamaWeights
    from oracle.synth import synth_weight
    from oracle.tensor_ref import OracleDevice, OracleTensor

    cname, wt_name, ct_name = WORKLOADS[workload]
    conf = getattr(R, cname)
    wt, ct = TYPE_ID[wt_name], TYPE_ID[ct_name]
    dim, hid, kv = conf.embedding_dim, conf.hidden_dim, conf.head_size() * conf.n_kv_heads
    # thread count: the reference takes it from the command line; use the count that is fastest for the dominant matvec on
    # this host (ascending, stop when it gets slower -- oversubscribed spin-waiting workers are pathological on big hosts)
    probe_w = synth_weight(wt, 2048, dim, SEED, 99, R.synth_scale(wt, dim))
    probe_x = np.random.default_rng(0).standard_normal(dim).astype(np.float32)
    threads, best = 1, float("inf")
    cpus = min(usable_cpus(), oc.hw_threads())
    for cand in sorted({c for c in (1, 2, 4, 8, 12, 16, 24, 32, 48, 64, 96, 128, cpus) if c <= cpus}):
        oc.gemv(wt, probe_w, 2048, dim, probe_x, threads=cand, flags=oc.ORDER_AVX2)
        dt = float("inf")
        for _ in range(3):                       # best of 3 batches of 5
            t0 = time.perf_counter()
            for _ in range(5):
                oc.gemv(wt, probe_w, 2048, dim, probe_x, threads=cand, flags=oc.ORDER_AVX2)
            dt = min(dt, time.perf_counter() - t0)
        if dt < best * 0.97:
            threads, best = cand, dt
        elif dt > best * 1.3:
            break
    dev = OracleDevice(thread_num=threads, flags=oc.ORDER_AVX2)
    n_sample_layers = min(sample_layers, conf.n_layers)

    def syn(rows, cols, t, tid):
        return OracleTensor.from_cpu(synth_weight(t, rows, cols, SEED, tid, R.synth_scale(t, cols)), [rows, cols], t, dev)
    rng = np.random.default_rng(SEED)

    def norm():
        return OracleTensor.from_cpu((1.0 + 0.05 * rng.standard_normal(dim)).astype(np.float32), [dim], oc.F32, dev)
    L = conf.n_layers
    w = dict(wq=[], wk=[], wv=[], wo=[], gate=[], up=[], down=[], ra=[], rf=[])
    for l in range(n_sample_layers):            # same tensor ids as crabml_b200.runner.synthetic_weights
        b = 7 * l
        w["wq"].append(syn(dim, dim, wt, b + 1)); w["wk"].append(syn(kv, dim, wt, b + 2)); w["wv"].append(syn(kv, dim, wt, b + 3))
        w["wo"].append(syn(dim, dim, wt, b + 4)); w["gate"].append(syn(hid, dim, wt, b + 5)); w["up"].append(syn(hid, dim, wt, b + 6))
        w["down"].append(syn(dim, hid, wt, b + 7)); w["ra"].append(norm()); w["rf"].append(norm())
    tok_embed = syn(conf.vocab_size, dim, wt, 7 * L + 1)
    out_w = syn(conf.vocab_size, dim, ct, 7 * L + 2)
    # REAL decode steps (warm-up, then `steps` timed tokens, mean) on two models cut from the same weights: 1 layer and
    # n_sample_layers layers (+ embedding, final norm, classifier).  A full token = the 1-layer token + (L - 1) x the per-layer
    # difference -- every layer of these shapes costs the same on the CPU (weights stream from DRAM once per token).
    times = {}
    for nl in sorted({1, n_sample_layers}):
        c = LlamaConfig(conf.n_heads, conf.n_kv_heads, nl, dim, hid, conf.seq_len, conf.vocab_size, conf.rms_norm_eps, conf.rope_dim or None)
        lw = LlamaWeights(tok_embed, w["wq"][:nl], w["wk"][:nl], w["wv"][:nl], w["wo"][:nl], w["gate"][:nl], w["down"][:nl], w["up"][:nl],
                          w["ra"][:nl], w["rf"][:nl], norm(), out_w)
        r = Llama2Runner(OracleTensor, c, lw, dev, warmup + steps + 8)
        pos = 0
        for i in range(warmup):
            r.forward([1 + i], pos); pos += 1
        t0 = time.perf_counter()
        for i in range(steps):
            r.forward([100 + i], pos); pos += 1
        times[nl] = (time.perf_counter() - t0) / max(1, steps)
    if n_sample_layers > 1:
        per_layer = (times[n_sample_layers] - times[1]) / (n_sample_layers - 1)
        if per_layer <= 0:                       # timer noise: split the sampled time by streamed bytes instead
            lb = 4 * R.weight_bytes(wt, dim, dim) + 3 * R.weight_bytes(wt, hid, dim)
            per_layer = times[n_sample_layers] * lb / (n_sample_layers * lb + R.weight_bytes(ct, conf.vocab_size, dim))
        rest = times[1] - per_layer
    else:
        per_layer, rest = times[1], 0.0
    per_token = per_layer * conf.n_layers + max(rest, 0.0)
    detail = {"layers_timed": n_sample_layers, "layers_model": conf.n_layers, "steps_timed": steps, "warmup_run": warmup,
              "ms_per_token_1_layer_model": times[1] * 1e3, f"ms_per_token_{n_sample_layers}_layer_model": times[n_sample_layers] * 1e3,
              "ms_per_layer": per_layer * 1e3, "extrapolated": n_sample_layers < conf.n_layers, "threads": threads, "usable_cpus": cpus,
              "hw_threads": oc.hw_threads(), "thread_probe": "ascending counts on a 2048-row matvec of the body type, fastest kept"}
    sample = (f"{steps} timed decode steps (after {warmup} warm-up) of a 1-layer and a {n_sample_layers}-layer cut of {workload} (same synthetic weights, seed "
              f"{SEED:#x}, embedding + final norm + classifier included); token time = 1-layer token + {conf.n_layers - 1} x per-layer difference; "
              f"AVX2-order C restatement of the reference, {threads} threads ({cpus} usable CPUs, {oc.hw_threads()} hardware threads)")
    return 1.0 / per_token, threads, sample, per_token, detail


def run_reference(args, rank, world):
    if rank != 0:
        return
    tps, threads, sample, per_token, detail = cpu_reference_tokens_per_s(args.workload, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": "decode_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_token * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int8", "data": "synthetic",
        "config": {"workload": f"{args.workload}-decode-synthetic", "note": "reference CPU path restated in C (oracle/): the Rust reference cannot be built here"},
        "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": threads, "kind": "port", "sample": sample, **detail},
        "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def write_outputs(directory: str, arrays: dict):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(directory, f"{name}.npy"), a.astype(np.float64 if a.dtype.kind in "iu" else np.float32))


def quick_decode(workload: str, local_rank: int, K: int, W: int, start_pos: int, outputs: dict | None = None):
    """Second measurement of the default run: the same decode loop (device-resident and e2e) for another weight type, so that one
    bench line covers the whole metric (Q8_0 AND Q4_0).  Returns a dict that is embedded in the main JSON line; `outputs`, when
    given, receives the logits of the last timed e2e step."""
    from crabml_b200 import CudaTensorDevice
    from crabml_b200 import runner as R
    cname, wt_name, ct_name = WORKLOADS[workload]
    conf = getattr(R, cname)
    wt, ct = TYPE_ID[wt_name], TYPE_ID[ct_name]
    dev = CudaTensorDevice(local_rank, lazy=2)
    try:
        weights = R.synthetic_weights(dev, conf, wt, ct, seed=SEED)
        runner = R.LlamaRunner(dev, conf, weights, min(conf.seq_len, start_pos + 2 * (W + K) + 8))
        bytes_per_token = runner.weight_bytes_per_token()
        pos, tok = 0, 1
        for _ in range(start_pos):
            runner.forward([tok], pos, export=False); pos += 1; tok = (tok * 7 + 3) % conf.vocab_size

        def step_e2e(t, p):
            lg = runner.forward([t], p, export=True)
            return int(np.flatnonzero(lg == lg.max())[-1])
        for _ in range(W):
            tok = step_e2e(tok, pos); pos += 1
        dev.synchronize()
        p0 = pos                                           # both timed regions decode at the same KV positions [p0, p0 + K)
        dev.timer_begin(); t0 = time.perf_counter()
        for _ in range(K):
            tok = step_e2e(tok, pos); pos += 1
        e2e_ms = max(dev.timer_end(), (time.perf_counter() - t0) * 1e3)
        if outputs is not None:
            outputs[f"{workload}_logits"] = runner.logits.copy()
        pos = p0
        l0 = dev.launch_count()
        dev.timer_begin()
        for i in range(K):
            runner.forward([(tok * 31 + 7 * i) % conf.vocab_size], pos, export=False); pos += 1
        val_ms = dev.timer_end()
        launches = dev.launch_count() - l0
        peaks, _ = measured_peaks()
        gbs = bytes_per_token / (val_ms / K * 1e-3) / 1e9
        out = {"workload": f"{workload}-decode-synthetic", "weights": wt_name, "classifier": ct_name, "value": K / (val_ms * 1e-3), "unit": "tok/s",
               "ms_per_step": val_ms / K, "e2e": {"value": K / (e2e_ms * 1e-3), "unit": "tok/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": conf.vocab_size * 4},
               "gpu_launches_device_resident": int(launches), "steps": K, "warmup": W,
               "roofline": {"bound": "hbm", "kernel": MEGA_NAMES.get(dev.mega_variant(), MEGA_NAMES[1])[0] if launches == K else "fused kernels (CUDA graph)", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": gbs / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": bytes_per_token, "frac_of_8TBs_nominal": gbs / 8000.0}}
        runner.close()
        return out
    finally:
        dev.close()


# --------------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    from crabml_b200 import CudaTensor, CudaTensorDevice
    from crabml_b200 import runner as R

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    sharded = world > 1 and args.multi == "sharded"

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v: float) -> float:
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    cname, wt_name, ct_name = WORKLOADS[args.workload]
    conf = getattr(R, cname)
    wt, ct = TYPE_ID[wt_name], TYPE_ID[ct_name]
    transport = args.comm
    lazy = args.lazy if not (sharded and transport == "nccl" and args.lazy == 2) else 1     # NCCL cannot run inside the megakernel
    dev = CudaTensorDevice(local_rank, lazy=lazy)
    plan = None
    if sharded:
        from crabml_b200 import sharding

        def exchange(blob):
            out = [None] * world
            dist.all_gather_object(out, blob)
            return out
        plan = sharding.make_plan(conf.n_heads, conf.n_kv_heads, conf.embedding_dim, conf.hidden_dim, conf.vocab_size, wt, rank, world)
        dev.init_comm(rank, world, exchange, transport)
    args.lazy = lazy
    weights = R.synthetic_weights(dev, conf, wt, ct, seed=SEED, plan=plan)
    K, W = args.steps, args.warmup
    kv_len = min(conf.seq_len, args.start_pos + 3 * (W + K) + 8)
    runner = R.LlamaRunner(dev, conf, weights, kv_len, plan=plan)
    bytes_per_token = runner.weight_bytes_per_token()

    # context: fill the KV cache up to start_pos with untimed steps so that decode runs at a realistic position
    pos, tok = 0, 1
    for _ in range(args.start_pos):
        runner.forward([tok], pos, export=False); pos += 1; tok = (tok * 7 + 3) % conf.vocab_size

    def step_e2e(t, p):
        lg = runner.forward([t], p, export=True)      # token id H2D (8 B) + logits D2H (vocab*4 B)
        return int(np.flatnonzero(lg == lg.max())[-1])   # sampler.rs:109-116 argmax (last max)

    for _ in range(W):
        tok = step_e2e(tok, pos); pos += 1
    # ---- timed region 1: e2e through the runner's public decode call with HOST buffers ---------------------------------------
    # ccr_runner_generate_greedy_ex: the prompt id goes host->device, the logits of EVERY step come device->host (pinned staging, async)
    # and the ids too; the host samples (argmax, sampler.rs:109-116) from those logits inside the timed region and must agree with the
    # device-side sampler that fed the next step.  No step waits for the host, so the GPU never idles between tokens.
    sampler = ClockSampler(local_rank); sampler.start()
    dev.synchronize(); barrier()
    p0 = pos              # every timed region decodes K tokens at the SAME KV positions [p0, p0 + K): the regions differ in how the host is involved, not in context length
    launches0 = dev.launch_count()
    dev.timer_begin(); t0 = time.perf_counter()
    tok_first = tok
    ids, lgs = runner.generate_greedy_logits([tok], K)
    host_ids = [int(np.flatnonzero(lg == lg.max())[-1]) for lg in lgs]
    e2e_ms_dev = dev.timer_end(); e2e_wall = time.perf_counter() - t0
    assert host_ids == ids and len(ids) == K, "host sampler and device sampler disagree"
    pos = p0; tok = tok_first                     # the synchronous variant reproduces the same greedy sequence
    launches_e2e = dev.launch_count() - launches0
    barrier()
    e2e_ms = max_over_ranks(max(e2e_ms_dev, e2e_wall * 1e3))      # host work (sampling) is part of e2e
    # the synchronous variant (one forward + blocking export + host argmax per token), for comparison
    dev.synchronize(); barrier()
    dev.timer_begin(); t0 = time.perf_counter()
    for _ in range(K):
        tok = step_e2e(tok, pos); pos += 1
    e2e_sync_ms = max_over_ranks(max(dev.timer_end(), (time.perf_counter() - t0) * 1e3))
    # what the callers of the two e2e regions received in the last step (the device-resident region exports nothing)
    outputs = {"logits": lgs[-1], "token_ids": ids, "logits_synchronous": runner.logits.copy()}
    pos = p0
    barrier()
    # ---- timed region 2: device-resident (no per-step host<->device traffic) -----------------------------------
    toks = [tok_first] + ids[:-1]          # the same K input tokens at the same positions as the e2e region: identical device work, no host round trips
    dev.synchronize(); barrier()
    launches1 = dev.launch_count()
    st0 = dev.lazy_stats() if args.lazy else None
    dev.timer_begin(); th0 = time.perf_counter()
    for i in range(K):
        runner.forward([toks[i]], pos, export=False); pos += 1
    host_issue_ms = (time.perf_counter() - th0) * 1e3          # host time to record+submit K tokens (GPU runs behind)
    val_ms = max_over_ranks(dev.timer_end())
    st1 = dev.lazy_stats() if args.lazy else None
    launches_val = dev.launch_count() - launches1
    clocks = sampler.stop()
    barrier()
    # the runner keeps no copy of the logits of an export=False step: repeat the region's last step (same token, same position,
    # same call) with the export, untimed
    outputs["logits_device_resident"] = runner.forward([toks[-1]], pos - 1, export=True).copy()

    # ---- roofline of the dominant kernel: ffn_gate/ffn_up-shaped matvec over all layers' weights (>> L2) ----------
    # (timed through an eager-mode device handle on the same GPU so that each matmul_vec is its own launch pair)
    m, k = weights["ffn_gate"][0].shape()
    dev.synchronize()
    edev = CudaTensorDevice(local_rank, lazy=False) if args.lazy else dev
    x = CudaTensor.new(np.random.default_rng(1).standard_normal(k).astype(np.float32), [k], edev)
    mats = [CudaTensor(wm.buf, wm.strider(), edev) for wm in weights["ffn_gate"] + weights["ffn_up"]]
    for wmat in mats[:4]:
        wmat.matmul_vec(x)
    reps = 3
    edev.synchronize()
    l0 = edev.launch_count()
    edev.timer_begin()
    for _ in range(reps):
        for wmat in mats:
            wmat.matmul_vec(x)
    mv_ms = edev.timer_end()
    n_mv = reps * len(mats)
    launches_per_mv = (edev.launch_count() - l0) / n_mv
    mv_bytes = R.weight_bytes(wt, m, k)
    mv_gbs = mv_bytes / (mv_ms / n_mv * 1e-3) / 1e9
    peaks, peak_src = measured_peaks()

    if rank == 0:
        streams = 1 if sharded or world == 1 else world       # sharded: ONE token stream over N GPUs; replicas: N streams
        value = streams * K / (val_ms * 1e-3)
        e2e = streams * K / (e2e_ms * 1e-3)
        if lazy == 2 and launches_val == K:
            # the dominant kernel IS the step: one mega_kernel launch per token streams every weight byte of this rank once
            mega_gbs = bytes_per_token / (val_ms / K * 1e-3) / 1e9
            mk_name, mk_file = MEGA_NAMES.get(dev.mega_variant(), MEGA_NAMES[1])
            roofline = {"bound": "hbm", "kernel": f"{mk_name} ({mk_file}): one persistent launch per decoded token, all matvec/attention/norm phases",
                        "achieved": mega_gbs, "peak": peaks["hbm_gbs"], "peak_source": peak_src, "unit": "GB/s", "frac": mega_gbs / peaks["hbm_gbs"],
                        "traffic": TRAFFIC.get((args.workload, world)), "traffic_source": "profiles/ (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if TRAFFIC.get((args.workload, world)) else None,
                        "algorithmic_bytes_per_launch": bytes_per_token, "us_per_launch": val_ms / K * 1e3, "frac_of_8TBs_nominal": mega_gbs / 8000.0}
        else:
            roofline = {"bound": "hbm", "kernel": f"matvec_stream_kernel<{wt_name}> {m}x{k} (+ activation quantize: {launches_per_mv:.0f} launches per matmul_vec)",
                        "achieved": mv_gbs, "peak": peaks["hbm_gbs"], "peak_source": peak_src, "unit": "GB/s",
                        "frac": mv_gbs / peaks["hbm_gbs"], "traffic": None, "algorithmic_bytes_per_launch": mv_bytes,
                        "us_per_launch": mv_ms / n_mv * 1e3, "frac_of_8TBs_nominal": mv_gbs / 8000.0}
        line = {
            "metric": "decode_tokens_per_s", "value": value, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": val_ms / K, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "int8",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}-decode-synthetic", "weights": wt_name, "classifier": ct_name, "kv_cache": "f32",
                       "start_pos": args.start_pos, "kv_positions": [int(p0), int(p0 + K)], "mode": "lazy: plan not megakernel-eligible (matvec types outside Q8_0/Q4_0 use the warp-per-row kernels): fused kernels, CUDA-graph replay" if (lazy == 2 and launches_val != K) else {0: "eager (one launch per trait call)", 1: "lazy: fused kernels, CUDA-graph replay", 2: "lazy: one persistent megakernel per token, CUDA-graph replay"}[args.lazy],
                       "multi_gpu": ("single GPU" if world == 1 else
                                     f"one token stream sharded over {world} GPUs: rows of wq/wk/wv/gate/up/classifier, block columns of wo/down; "
                                     f"exchange = {'one-shot NVLink peer stores fused into the megakernel' if transport == 'p2p' and lazy == 2 else 'one-shot NVLink peer-store kernel' if transport == 'p2p' else 'ncclAllReduce/ncclAllGather'} "
                                     f"(2 allreduce of [dim] f32 per layer + 1 allgather of logits)" if sharded else f"{world} independent replicas"),
                       "weight_bytes_per_token_per_gpu": bytes_per_token,
                       "l2_policy": f"weights streamed once per token ({bytes_per_token / 1e9:.2f} GB >> 126 MB L2): inputs larger than L2",
                       "weight_bytes_per_token": bytes_per_token,
                       "hbm_frac_whole_step": bytes_per_token / (val_ms / K * 1e-3) / 1e9 / peaks["hbm_gbs"]},
            "e2e": {"value": e2e, "unit": "tok/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": conf.vocab_size * 4 + 8,
                    "ms_per_step": e2e_ms / K,
                    "api": "ccr_runner_generate_greedy_ex: sampling on the device feeds the next step, logits + ids exported asynchronously every step, host argmax checked in the timed region",
                    "synchronous_variant": {"value": streams * K / (e2e_sync_ms * 1e-3), "unit": "tok/s", "api": "ccr_runner_forward + blocking export + host argmax per token"}},
            "gpu_launches": int(launches_e2e),
            "gpu_launches_device_resident": int(launches_val),
            "roofline": roofline,
            "roofline_matvec_eager": {"kernel": f"matvec_stream_kernel<{wt_name}> {m}x{k} + activation quantize ({launches_per_mv:.0f} launches per matmul_vec, eager handle, not in the timed region)",
                                      "achieved": mv_gbs, "unit": "GB/s", "frac": mv_gbs / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": mv_bytes,
                                      "us_per_launch": mv_ms / n_mv * 1e3},
            "clocks": clocks,
            "lazy_stats": dev.lazy_stats() if args.lazy else None,
            "host_ms_per_step": {"issue_total": host_issue_ms / K,
                                 **({k: (st1[k] - st0[k]) / 1e3 / K for k in ("host_us_record", "host_us_fuse", "host_us_submit")} if args.lazy else {})},
        }
        if world == 1 and not args.no_cpu_baseline:
            tps, threads, sample, _, detail = cpu_reference_tokens_per_s(args.workload, steps=min(K, 8), warmup=2)
            line["cpu_baseline"] = {"value": tps, "unit": "tok/s", "cores": threads, "kind": "port", "sample": sample, **detail}
    runner.close()
    dev.close()
    if rank == 0:
        if world == 1 and args.workload == "llama2-7b-q8_0" and not args.no_also:
            # the metric names Q8_0 AND Q4_0: same loop, same shapes, Q4_0 blocks (llama.cpp-style Q4_0 files keep a Q6_K classifier:
            # run `--workload llama2-7b-q4_0-q6k` for that variant)
            weights = None
            try:
                line["also"] = {"llama2-7b-q4_0": quick_decode("llama2-7b-q4_0", local_rank, K, W, args.start_pos, outputs)}
            except Exception as e:      # the second block must never cost the main line
                line["also"] = {"llama2-7b-q4_0": {"error": repr(e)}}
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()



def run_prefill(args, rank, world, local_rank):
    """BASELINE.json config 5: every matmul_vec of a `--prefill-tokens`-token prompt pass (Tensor::matmul_vec with a (b, k) rhs) on the
    tensor-core path: per layer wq, wk, wv, wo, ffn_gate, ffn_up, ffn_down on (b, k) activations, then the classifier on the last row.
    A step = all 225 matmuls once.  This is the DENSE part of a prefill (58 of ~63 TFLOP for Mistral-7B at 4096 tokens); attention,
    norms and RoPE of a batched forward are not part of this workload (the reference has no batched forward: llama2.rs:111-139 walks
    the prompt token by token)."""
    from crabml_b200 import CudaTensor, CudaTensorDevice
    from crabml_b200 import runner as R
    if rank != 0:
        return
    cname, wt_name, ct_name = WORKLOADS[args.workload]
    conf = getattr(R, cname)
    wt, ct = TYPE_ID[wt_name], TYPE_ID[ct_name]
    b = args.prefill_tokens
    dev = CudaTensorDevice(local_rank, lazy=0)
    weights = R.synthetic_weights(dev, conf, wt, ct, seed=SEED)
    dim, hid = conf.embedding_dim, conf.hidden_dim
    rng = np.random.default_rng(SEED)
    x_dim = CudaTensor.new(rng.standard_normal(b * dim).astype(np.float32), [b, dim], dev)
    x_hid = CudaTensor.new(rng.standard_normal(b * hid).astype(np.float32), [b, hid], dev)
    x_last = CudaTensor.new(rng.standard_normal(dim).astype(np.float32), [dim], dev)
    flops = 0
    for key, kk in (("wq", dim), ("wk", dim), ("wv", dim), ("wo", dim), ("ffn_gate", dim), ("ffn_up", dim), ("ffn_down", hid)):
        for t in weights[key]:
            flops += 2 * b * t.shape()[0] * kk
    wbytes = sum(R.weight_bytes(t.dtype(), *t.shape()) for key in ("wq", "wk", "wv", "wo", "ffn_gate", "ffn_up", "ffn_down") for t in weights[key])

    def step():
        """-> classifier output and the outputs of the last layer's seven GEMMs (the other layers' are dropped at once)."""
        for l in range(conf.n_layers):
            last = {key: weights[key][l].matmul_vec(x_dim) for key in ("wq", "wk", "wv", "wo", "ffn_gate", "ffn_up")}
            last["ffn_down"] = weights["ffn_down"][l].matmul_vec(x_hid)
        return weights["output_weight"].matmul_vec(x_last), last
    K, W = args.steps, args.warmup
    for _ in range(W):
        step()
    sampler = ClockSampler(local_rank); sampler.start()
    dev.synchronize()
    l0 = dev.launch_count()
    dev.timer_begin()
    for _ in range(K):
        logits, gemms = step()
    ms = dev.timer_end()
    launches = dev.launch_count() - l0
    # e2e: what crosses the host boundary in a prompt pass -- the token ids go host->device (the embedding rows are gathered on the
    # device, llama2.rs:223-224), the logits of the last position come back
    ids = [int(v) for v in rng.integers(0, conf.vocab_size, b)]
    from crabml_b200 import capi as _capi
    dev.synchronize()
    dev.timer_begin(); t0 = time.perf_counter()
    for _ in range(K):
        xd = CudaTensor.alloc([b, dim], _capi.F32, dev)
        xd.copy_rows_from(weights["token_embed"], ids)
        for l in range(conf.n_layers):
            for key in ("wq", "wk", "wv", "wo", "ffn_gate", "ffn_up"):
                weights[key][l].matmul_vec(xd)
            weights["ffn_down"][l].matmul_vec(x_hid)
        weights["output_weight"].matmul_vec(x_last).export()
    e2e_ms = max(dev.timer_end(), (time.perf_counter() - t0) * 1e3)
    clocks = sampler.stop()
    peaks, peak_src = measured_peaks()
    tf = flops / (ms / K * 1e-3) / 1e12
    peak_tf = peaks.get("bf16_tflops_sustained", 1431.9)
    line = {"metric": "prefill_tokens_per_s", "value": b * K / (ms * 1e-3), "unit": "tok/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 operand tiles (dequantised Q8_0 weights, quantised activations), f32 accumulate",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}-dense-matmuls-synthetic", "prompt_tokens": b, "weights": wt_name,
                       "scope": "the 225 matmul_vec calls of a prompt pass (per-call activation quantisation and weight dequantisation included); attention / norms / RoPE of a "
                                "batched forward are not part of this workload",
                       "l2_policy": f"{wbytes / 1e9:.2f} GB of weights and {b * hid * 4 / 1e6:.0f} MB activations per step: inputs larger than L2",
                       "flop_per_step": flops},
            "e2e": {"value": b * K / (e2e_ms * 1e-3), "unit": "tok/s", "h2d_bytes_per_step": b * 8, "d2h_bytes_per_step": conf.vocab_size * 4, "ms_per_step": e2e_ms / K},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "umma_gemm_kernel (prefill_gemm.cu): TMA -> smem ring -> tcgen05.mma kind::f16 -> TMEM -> tcgen05.ld epilogue",
                         "achieved": tf, "peak": peak_tf, "peak_source": peak_src + " bf16_tflops_sustained", "unit": "TFLOP/s", "frac": tf / peak_tf, "traffic": None,
                         "note": "whole step (dequantise + quantise + GEMM launches) over the dense FLOPs; the GEMM kernel alone is profiled in profiles/"},
            "clocks": clocks}
    if args.dump_outputs:
        pick = np.random.default_rng(SEED)          # the same 4096 elements of each [b, rows] product in every run
        write_outputs(args.dump_outputs, {"logits": logits.export(),
                                          **{f"{key}_sample": y.export()[np.sort(pick.choice(b * y.shape()[1], 4096, replace=False))]
                                             for key, y in gemms.items()}})
    print(json.dumps(line))
    dev.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="llama2-7b-q8_0", choices=sorted(WORKLOADS))
    ap.add_argument("--start-pos", type=int, default=32, help="KV-cache length before the timed decode steps")
    ap.add_argument("--lazy", type=int, default=2, help="2 = record+fuse, one persistent megakernel per token (default); 1 = fused kernels in a CUDA graph; 0 = one launch per trait call")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--prefill-tokens", type=int, default=4096)
    ap.add_argument("--no-also", action="store_true", help="skip the second (Q4_0) measurement of the default run")
    ap.add_argument("--multi", default="sharded", choices=["sharded", "replicas"], help="N > 1: shard one token stream (strong scaling, default) or run N independent replicas")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"], help="exchange transport of the sharded path: one-shot NVLink peer stores (default) or the NCCL baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload.endswith("-prefill"):
        run_prefill(args, rank, world, local_rank)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
