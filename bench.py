#!/usr/bin/env python
"""Benchmark of the SuDoRM-RF forward path (BASELINE.json metric: mixtures/sec,
4 s @ 8 kHz, 2 sources).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repo's kernels)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm (CPU oracle port)

One "step" = one forward pass of the separator over one synthetic batch.  At
N > 1 the batch is sharded by giving every rank its own batch of the same size
(weak scaling, no collective inside the step; the packed weights are broadcast
ONCE with NCCL before timing).  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

# BASELINE.json configs (SURVEY.md §8 shapes).  The headline / default workload is
# configs[1]: Improved SuDoRM-RF U16/512, batch 32 x 4 s @ 8 kHz on one B200.
WORKLOADS = {
    "improved_u16_512": dict(variant="improved", B=32, T=32000, kw=dict(
        out_channels=256, in_channels=512, num_blocks=16, upsampling_depth=5,
        enc_kernel_size=21, enc_num_basis=512, num_sources=2)),
    "improved_u8_512": dict(variant="improved", B=1, T=32000, kw=dict(
        out_channels=256, in_channels=512, num_blocks=8, upsampling_depth=5,
        enc_kernel_size=21, enc_num_basis=512, num_sources=2)),
    "improved_u36_2048": dict(variant="improved", B=64, T=32000, kw=dict(
        out_channels=512, in_channels=512, num_blocks=36, upsampling_depth=6,
        enc_kernel_size=21, enc_num_basis=2048, num_sources=2)),
    "groupcomm_u8_512": dict(variant="groupcomm", B=16, T=32000, kw=dict(
        out_channels=256, in_channels=512, num_blocks=8, upsampling_depth=5,
        enc_kernel_size=21, enc_num_basis=512, num_sources=2, group_size=16)),
    "improved_u36_4096_16k": dict(variant="improved", B=32, T=64000, kw=dict(
        out_channels=512, in_channels=512, num_blocks=36, upsampling_depth=6,
        enc_kernel_size=21, enc_num_basis=4096, num_sources=2)),
    # SURVEY 8f.3 sibling variant (not a BASELINE config): CausalSuDORMRF with its constructor defaults
    # (causal_improved_sudormrf_v3.py:121-129) at the headline batch / length
    "causal_u16_512": dict(variant="causal", B=32, T=32000, kw=dict(
        in_audio_channels=1, out_channels=128, in_channels=512, num_blocks=16, upsampling_depth=4,
        enc_kernel_size=21, enc_num_basis=512, num_sources=2)),
    # SURVEY 8f.3 sibling variant (not a BASELINE config): the ORIGINAL SuDoRM-RF with its constructor defaults
    # (sudormrf.py:186-193) at the headline batch / length
    "original_u16_512": dict(variant="original", B=32, T=32000, kw=dict(
        out_channels=128, in_channels=512, num_blocks=16, upsampling_depth=4,
        enc_kernel_size=21, enc_num_basis=512, num_sources=2)),
}


def model_class(variant):
    import sudo_rm_rf_b200 as P
    return {"improved": P.SuDORMRF, "groupcomm": P.GroupCommSudoRmRf, "causal": P.CausalSuDORMRF,
            "original": P.OriginalSuDORMRF}[variant]
METRIC = "mixtures_per_sec_forward_4s_8kHz_2src"
UNIT = "mixtures/s"
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, name, t):
    """Writes the output `t` ([batch, ...]) as out_dir/<name>.npy in float32.  Above DUMP_LIMIT_BYTES only a fixed,
    seeded sample of its batch rows (in batch order) is written, so runs with the same arguments write the same rows."""
    import numpy as np
    t = t.detach().float().cpu()
    row_bytes = 4 * t[0].numel()
    if t.numel() * 4 > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // row_bytes)
        rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        t = t[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Dense bf16 TFLOP/s (cuBLAS, burst) measured on this pool's B200s; fallback: the profiling guide's figure."""
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        if "bf16_tflops" in p:
            return float(p["bf16_tflops"]), "measured (MEASURED_PEAKS.json, burst)"
    return 1670.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------
# algorithmic bytes / flops model (SURVEY.md §8d), fp32, every intermediate
# written once and read once
# --------------------------------------------------------------------------
def algorithmic_model(w):
    kw = w["kw"]
    N, Co, Ci = kw["enc_num_basis"], kw["out_channels"], kw["in_channels"]
    U, D, S, K = kw["num_blocks"], kw["upsampling_depth"], kw["num_sources"], kw["enc_kernel_size"]
    hop = K // 2
    q = hop * 2 ** D
    Tp = max(q, -(-w["T"] // q) * q)
    L = Tp // hop
    kappa = 5 + sum(2.0 ** -(d - 1) + 2.0 ** -d for d in range(1, D)) + sum(2.0 ** -d for d in range(D))
    a_blk = 4 * L * (3 * Co + kappa * Ci)
    if w["variant"] == "causal":
        # no normalisation layers: the depthwise stage is one local pass, so the model is the fused schedule's own
        # minimum (x read, y written + read, m written + read, residual read, x written), not the level-by-level one
        a_blk = 4 * L * (3 * Co + 4 * Ci)
        a_mix = 4 * (Tp + 2 * N * L + Co * L) + U * a_blk + 4 * (Co * L + S * Tp)
        flops = 2 * L * (K * N + N * Co + U * (2 * Co * Ci + 11 * Ci * (2 - 2.0 ** (1 - D))) + Co * S * N + K * S * S * N)
        return dict(L=L, Tp=Tp, a_blk=a_blk, a_mix=a_mix, flops=flops,
                    res_bytes=4 * L * (Ci + 2 * Co), res_flops=2 * Co * Ci * L)
    if w["variant"] == "original":
        # sudormrf.py: lcm padding; per block two more [Co, L] tensors than the improved block (conv_1x1_exp output
        # written + read, the residual sum written and read by two consumers): 5 Co instead of 3 Co; the back end
        # is modelled like the improved one (block output + encoder output in, S waveforms out)
        import math
        q = hop * 2 ** D // math.gcd(hop, 2 ** D)
        Tp = w["T"] if w["T"] % q == 0 else w["T"] + q - w["T"] % q
        L = Tp // hop
        a_blk = 4 * L * (5 * Co + kappa * Ci)
        a_mix = 4 * (Tp + 2 * N * L + Co * L) + U * a_blk + 4 * (Co * L + N * L + S * Tp)
        flops = 2 * L * (K * N + N * Co + U * (2 * Co * Ci + 5 * Ci * (2 - 2.0 ** (1 - D))) +
                         (Co * N if Co != N else 0) + N * S * N + K * S * N)
        return dict(L=L, Tp=Tp, a_blk=a_blk, a_mix=a_mix, flops=flops,
                    res_bytes=4 * L * (Ci + Co), res_flops=2 * Co * Ci * L)
    gc = w["variant"] == "groupcomm"
    if gc:
        a_blk += 4 * L * 4 * Co
    a_front = 4 * (Tp + 2 * N * L + Co * L)
    a_back = 4 * (Co * L + N * L + S * Tp)
    a_mix = a_front + U * a_blk + a_back
    G = kw.get("group_size", 1) if gc else 1
    gemm = 2 * Co * Ci / G
    flops = 2 * L * (K * N + N * Co + U * (gemm + 5 * Ci * (2 - 2.0 ** (1 - D))) + Co * S * N + K * S * S * N)
    if gc:
        n = Co // G
        H = 3 * n
        flops += U * 2 * L * (3 * G * n * H + H * H)
    return dict(L=L, Tp=Tp, a_blk=a_blk, a_mix=a_mix, flops=flops,
                res_bytes=4 * L * (Ci + 2 * Co), res_flops=2 * Co * Ci * L / G)


# --------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md)
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [s.strip() for s in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------
# reference arm / cpu baseline: the CPU oracle port of the reference forward
# --------------------------------------------------------------------------
def host_cores():
    """(logical CPUs visible to this process, physical cores)."""
    logical = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = logical
    return logical, physical


def cpu_forward_rate(w, sample_B, steps, warmup, budget_s=None):
    """mixtures/s of the CPU oracle port (same torch op sequence as the reference's forward,
    improved_sudormrf.py:283-301) on ALL host cores.  Protocol of BASELINE.md section 2 / the reference's notebook
    (sudormrf_extract_computation_metrics_example.ipynb:125-146): batch 1, >= 10 repetitions, median.
    torchrun exports OMP_NUM_THREADS=1 per rank, so the thread count is set explicitly."""
    from oracle import sudormrf_oracle as O
    logical, physical = host_cores()
    # one thread per PHYSICAL core: with one per logical CPU (SMT) the GlobLN passes of the port ran 40x slower
    # on the 64-core / 128-thread box (80 s per forward instead of ~0.3-0.6 s)
    torch.set_num_threads(max(1, min(logical, physical)))
    cfg = O.Config(variant=w["variant"], **w["kw"])
    sd = O.make_state_dict(cfg, seed=0, perturbed=False)
    x = torch.rand(sample_B, 1, w["T"], generator=torch.Generator().manual_seed(1))
    times = []
    with torch.no_grad():
        for _ in range(warmup):
            O.forward(cfg, sd, x)
        t_start = time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter()
            y = O.forward(cfg, sd, x)
            times.append(time.perf_counter() - t0)
            if budget_s is not None and time.perf_counter() - t_start > budget_s and len(times) >= 3:
                break
    times.sort()
    med = times[len(times) // 2]
    return {"rate": sample_B / med, "sec_per_step": med, "done": len(times), "threads": torch.get_num_threads(),
            "logical_cpus": logical, "physical_cores": physical, "best": sample_B / times[0], "last_output": y}


def run_reference(args, w, wl_name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_B = 1
    r = cpu_forward_rate(w, sample_B, args.steps, max(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "estimates", r["last_output"])
    line = {
        "impl": "reference", "metric": METRIC, "value": r["rate"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["done"], "warmup": max(args.warmup, 1), "ms_per_step": r["sec_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (torch.rand mixtures, default-init weights)",
        "config": {"workload": wl_name, "batch_per_step": sample_B, "samples": w["T"],
                   "note": "CPU arm = this repo's oracle PORT of the reference forward (oracle/sudormrf_oracle.py: the same "
                           "torch op sequence, pinned bit-exactly to reference-generated goldens); it is NOT the unmodified "
                           "reference module, which is not shipped to the GPU box.  Batch 1, median over the steps, all host "
                           "cores (BASELINE.md section 2 protocol); under torchrun only rank 0 runs."},
        "cpu_baseline": {"value": r["rate"], "unit": UNIT, "cores": r["threads"], "physical_cores": r["physical_cores"],
                         "kind": "port", "best": r["best"],
                         "sample": f"median of {r['done']} forwards of batch {sample_B} x {w['T']} samples"},
        "e2e": {"value": r["rate"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------
def run_b200(args, w, wl_name):
    import ctypes as C
    import torch.distributed as dist
    import sudo_rm_rf_b200 as P
    from sudo_rm_rf_b200 import _engine, _native
    from oracle import sudormrf_oracle as O      # weights generator + cpu_baseline leg only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (B200 arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B, T = (args.batch or w["B"]), w["T"]
    model = model_class(w["variant"])(**w["kw"])
    cfg_o = O.Config(variant=w["variant"], **w["kw"])
    if rank == 0:
        model.load_state_dict(O.make_state_dict(cfg_o, seed=0, perturbed=False))
    model = model.to(dev).eval()
    if world > 1:
        # ONE broadcast of all weights over NVLink (NCCL), outside the timed step; the step itself
        # has no collective: every rank separates its own shard of the batch
        from sudo_rm_rf_b200 import sharding
        sharding.broadcast_parameters(model, src=0)
    cfg = _engine.make_config(model)
    launches_per_step = _native.lib().sdr_forward_launch_count_at(C.byref(cfg), w["T"])

    g = torch.Generator().manual_seed(1234 + rank)
    host_x = torch.rand(B, 1, T, generator=g).pin_memory()      # the reference's bench input (notebook :128)
    x = host_x.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    stream = torch.cuda.Stream(device=dev)
    with torch.no_grad(), torch.cuda.stream(stream):
        y = model(x)                      # packs weights, sizes the workspace
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            y = model(x)
        for _ in range(max(args.warmup, 3)):
            graph.replay()
        stream.synchronize()

        def barrier():
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)

        # ---- device-resident timing: K graph replays, L2 flushed between steps ----
        sampler = ClockSampler(local) if rank == 0 else None
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(args.steps)]
        barrier()
        if sampler:
            sampler.start()
        wall0 = time.perf_counter()
        for s, e in evs:
            flush.fill_(1)
            s.record(stream)
            graph.replay()
            e.record(stream)
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if sampler else None
        dev_ms = sum(s.elapsed_time(e) for s, e in evs)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, "estimates", y)      # the last timed replay's separated sources

        # ---- end to end: pinned host mixtures in, pinned host estimates out, every step ----
        host_y = torch.empty(B, w["kw"]["num_sources"], T).pin_memory()
        for _ in range(3):
            model.forward_host(host_x, host_y)
        stream.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            model.forward_host(host_x, host_y)
            stream.synchronize()           # the step's result is read on the host
        e1.record(stream)
        barrier()
        e2e_ms = e0.elapsed_time(e1)

        # ---- every kernel of a U-ConvBlock alone + the block as a whole (CUDA events on the launching stream) ----
        roof = None
        lat1 = None
        if rank == 0:
            roof = roofline_block(w, B, stream, flush, dev)
            lat1 = latency_b1(model, w, dev, stream)

    # ---- the other BASELINE configs, short runs on every rank (so the 8-GPU scaling run yields their figures too) ----
    others = []
    other_ms = []
    if wl_name == "improved_u16_512" and not args.no_other_configs:
        del graph
        torch.cuda.empty_cache()
        for name in ("improved_u36_2048", "groupcomm_u8_512", "improved_u36_4096_16k", "causal_u16_512",
                     "original_u16_512"):
            ow, ms, n_par = short_config_run(name, dev, stream, flush)
            others.append((name, ow, n_par))
            other_ms.append(ms)

    t = torch.tensor([dev_ms, e2e_ms] + other_ms, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, *other_ms = t.tolist()

    if rank == 0:
        peak, peak_src = load_peaks()
        am = algorithmic_model(w)
        n_params = sum(p.numel() for p in model.parameters())
        total_mix = B * world * args.steps
        value = total_mix / (dev_ms / 1e3)
        fwd_bytes = B * am["a_mix"] + 4 * n_params
        fwd_gbs = fwd_bytes / (dev_ms / args.steps / 1e3) / 1e9
        eager = None
        if world == 1:      # comparators are timed at N=1 only
            eager = eager_cuda_rate(w, B, dev)
            r = cpu_forward_rate(w, 1, steps=30, warmup=1, budget_s=15.0)
            cpu_baseline = {"value": r["rate"], "unit": UNIT, "cores": r["threads"], "physical_cores": r["physical_cores"],
                            "kind": "port", "best": r["best"],
                            "sample": f"median of {r['done']} forwards of batch 1 x {T} samples "
                                      f"({r['sec_per_step']:.2f} s each), same model, oracle port of the reference forward"}
        else:
            cpu_baseline = None
        other_configs = []
        for (name, ow, n_par), ms in zip(others, other_ms):
            oam = algorithmic_model(ow)
            ob = ow["B"] * oam["a_mix"] + 4 * n_par
            other_configs.append({"workload": name, "batch_per_gpu": ow["B"], "global_batch": ow["B"] * world,
                                  "samples": ow["T"], "steps": 5, "ms_per_step": ms,
                                  "value": ow["B"] * world / (ms / 1e3), "unit": UNIT,
                                  "forward_hbm_frac": ob / (ms / 1e3) / 1e9 / peak})
            if ow["variant"] == "causal":      # the sibling variant's own kernels, each alone and as one block
                ck, cpb, _, _ = time_block(ow, ow["B"], stream, flush, dev)
                other_configs[-1]["kernels"] = ck
                other_configs[-1]["per_block"] = cpb
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (torch.rand mixtures, default-init weights)",
            "config": {"workload": wl_name, "batch_per_gpu": B, "global_batch": B * world,
                       "samples": T, "sources": w["kw"]["num_sources"], "parallelism": f"dp{world}",
                       "l2": "256 MiB flush write between timed steps; one step streams "
                             f"{fwd_bytes / 1e9:.1f} GB (algorithmic) through a >1 GB workspace >> 126 MB L2",
                       "timing": "CUDA events around each CUDA-graph replay, summed over K steps, max over ranks",
                       "wall_s_timed_loop": wall},
            "e2e": {"value": total_mix / (e2e_ms / 1e3), "unit": UNIT,
                    "h2d_bytes_per_step": B * T * 4 * world,
                    "d2h_bytes_per_step": B * w["kw"]["num_sources"] * T * 4 * world,
                    "api": "model.forward_host (sdr_forward_host): pinned host in/out, sync per step"},
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step,
            "clocks": clocks,
            "roofline": roof,
            "forward_hbm": {"algorithmic_bytes_per_step": fwd_bytes, "achieved": fwd_gbs, "peak": peak,
                            "unit": "GB/s", "frac": fwd_gbs / peak, "peak_source": peak_src,
                            "gflop_per_mixture": am["flops"] / 1e9},
            "cpu_baseline": cpu_baseline,
            "eager_cuda_baseline": eager,
            "other_configs": other_configs,
            "latency_b1": lat1,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------
# per-kernel and per-U-ConvBlock timing through the stage-level C-ABI entry points
# --------------------------------------------------------------------------
def arrD_(ts, D):
    import ctypes as C
    return (C.c_void_p * D)(*[t.data_ptr() for t in ts])


def block_launchers(w, B, dev, stream):
    """The 3 + D kernels of ONE U-ConvBlock at the workload's shapes, in forward order, as
    [(name, launch, algorithmic_bytes, flops)], operating on synthetic tensors through the stage-level C-ABI
    (the same entry points `sdr_forward` dispatches to).  Returns (launchers, keepalive)."""
    import ctypes as C
    from sudo_rm_rf_b200 import _native as N
    lib = N.lib()
    kw = w["kw"]
    gc = w["variant"] == "groupcomm"
    G = kw.get("group_size", 1) if gc else 1
    am = algorithmic_model(w)
    L, D = am["L"], kw["upsampling_depth"]
    S, Co, Ci = B * G, kw["out_channels"] // G, kw["in_channels"] // G
    sp = C.c_void_p(stream.cuda_stream)
    P = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *shape: torch.randn(*shape, device=dev, generator=gen)
    ones, zeros = torch.ones(max(Ci, Co), device=dev), torch.zeros(max(Ci, Co), device=dev)
    slope = torch.full((1,), 0.25, device=dev)
    keep = [ones, zeros, slope]

    def stats_of(t):
        td = t.double().reshape(t.shape[0], -1)
        return torch.stack([td.sum(1), (td * td).sum(1)], 1).contiguous()

    x = rn(S, Co, L)                      # block input == residual stream (updated in place by res_conv)
    y = torch.empty(S, Ci, L, device=dev)
    z = [torch.empty(S, Ci, L >> d, device=dev) for d in range(D)]
    st = [torch.zeros(S, 2, dtype=torch.float64, device=dev) for _ in range(D + 2)]
    keep += [x, y, z, st]
    out = []

    def gemm(name, xin, nin, M, K, res, yout, stats):
        Wt = rn(M, K) / K ** 0.5
        bias = rn(M)
        nbytes = lib.sdr_pointwise_mma_packed_bytes(M, K)
        keep.extend([Wt, bias])
        if nbytes:
            wpk = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            N.check(lib.sdr_pointwise_mma_pack(P(Wt), M, K, P(wpk), sp))
            keep.append(wpk)
            fn = lambda: N.check(lib.sdr_pointwise_mma(P(xin), C.byref(nin), P(wpk), P(bias), P(res), P(None), 0,
                                                       P(yout), P(stats), S, M, K, L, 0, sp))
            return name + " [pw_mma_kernel tcgen05 bf16x3]", fn
        fn = lambda: N.check(lib.sdr_pointwise(P(xin), C.byref(nin), P(Wt), P(bias), P(res), P(None), 0,
                                               P(yout), P(stats), S, M, K, L, 0, sp))
        return name + " [pw_gemm_kernel FFMA]", fn

    none = N.SdrNormIn(0, 0, 0, 0, 1.0)
    keep.append(none)
    if w["variant"] == "causal":
        # causal block (causal_improved_sudormrf_v3.py:98-118): proj GEMM, the whole depthwise stage in one pass,
        # res_conv (gain folded into its weights) + in-place skip connection; no statistics anywhere
        n_, f_ = gemm("proj_1x1", x, none, Ci, Co, None, y, None)
        out.append((n_, f_, 4 * L * S * (Co + Ci), 2.0 * Co * Ci * L * S))
        w21, b21 = [rn(Ci, 1, 21) * 0.3 for _ in range(D)], [rn(Ci) for _ in range(D)]
        slopes = [slope] * D
        wa, ba, sa = arrD_(w21, D), arrD_(b21, D), arrD_(slopes, D)
        keep.extend([w21, b21, wa, ba, sa])
        out.append((f"causal depthwise stage: PReLU, {D} masked 21-tap levels, up-sample + add, one pass [causal_pyramid_kernel]",
                    lambda: N.check(lib.sdr_causal_pyramid(P(y), P(slope), wa, ba, sa, P(z[0]), D, S, Ci, L, sp)),
                    4 * S * Ci * 2 * L, 22.0 * Ci * S * sum(L >> d for d in range(D))))
        n_, f_ = gemm("res_conv+skip", z[0], none, Co, Ci, x, x, None)
        out.append((n_, f_, 4 * L * S * (Ci + 2 * Co), 2.0 * Co * Ci * L * S))
        return out, (lambda: None), keep
    # proj_1x1: raw residual stream in, raw y + statistics out
    n_, f_ = gemm("proj_1x1", x, none, Ci, Co, None, y, st[0])
    out.append((n_, f_, 4 * L * S * (Co + Ci), 2.0 * Co * Ci * L * S))
    arrD = lambda ts: (C.c_void_p * D)(*[t.data_ptr() for t in ts])
    w5s, b5s = [rn(Ci, 5) for _ in range(D)], [rn(Ci) for _ in range(D)]
    keep.extend([w5s, b5s])
    nin0 = N.SdrNormIn(st[0].data_ptr(), ones.data_ptr(), zeros.data_ptr(), slope.data_ptr(), float(Ci * L))
    keep.append(nin0)
    scratch_bytes = lib.sdr_pyramid_scratch_bytes(S, Ci, D, L)
    level_bytes = 4 * S * Ci * (2 * L + sum((L >> (d - 1)) + (L >> d) for d in range(1, D)))
    merge_bytes = 4 * S * Ci * (L + sum(L >> d for d in range(D)))
    if scratch_bytes:
        # the forward's path at this shape: every depthwise level in ONE pass over y, then the affine merge
        scratch = torch.empty(scratch_bytes, dtype=torch.uint8, device=dev)
        wa, ba, ga, bea, za = arrD(w5s), arrD(b5s), arrD([ones] * D), arrD([zeros] * D), arrD(z)
        keep.extend([scratch, wa, ba, ga, bea, za])
        out.append((f"depthwise pyramid, levels 0..{D - 1} in one pass (+ GlobLN solve)",
                    lambda: N.check(lib.sdr_depthwise_pyramid(P(y), C.byref(nin0), wa, ba, ga, bea, za, P(st[1]), P(scratch),
                                                              D, S, Ci, L, sp)),
                    level_bytes, 10.0 * Ci * S * sum(L >> d for d in range(D))))
        out.append(("merge (affine in the raw levels)",
                    lambda: N.check(lib.sdr_merge_pyramid(za, P(scratch), D, P(y), P(st[D + 1]), S, Ci, L, sp)),
                    merge_bytes, 3.0 * D * Ci * L * S))
    else:
        for d in range(D):
            src = y if d == 0 else z[d - 1]
            Lin = L if d == 0 else L >> (d - 1)
            nin = nin0 if d == 0 else N.SdrNormIn(st[d].data_ptr(), ones.data_ptr(), zeros.data_ptr(), 0, float(Ci * Lin))
            keep.append(nin)
            stride = 1 if d == 0 else 2
            out.append((f"depthwise level {d} (stride {stride})",
                        (lambda src=src, nin=nin, d=d, Lin=Lin, stride=stride: N.check(lib.sdr_depthwise(
                            P(src), C.byref(nin), P(w5s[d]), P(b5s[d]), P(z[d]), P(st[d + 1]), S, Ci, Lin, stride, sp))),
                        4 * S * Ci * (Lin + (L >> d)), 10.0 * Ci * (L >> d) * S))
        fins = (N.SdrNormIn * D)(*[N.SdrNormIn(st[d + 1].data_ptr(), ones.data_ptr(), zeros.data_ptr(), 0,
                                               float(Ci * (L >> d))) for d in range(D)])
        zp = arrD(z)
        keep.extend([fins, zp])
        out.append(("merge", lambda: N.check(lib.sdr_merge(zp, fins, D, P(y), P(st[D + 1]), S, Ci, L, sp)),
                    merge_bytes, 3.0 * D * Ci * L * S))
    # res_conv + in-place skip connection
    nf = N.SdrNormIn(st[D + 1].data_ptr(), ones.data_ptr(), zeros.data_ptr(), slope.data_ptr(), float(Ci * L))
    keep.append(nf)
    n_, f_ = gemm("res_conv+skip", y, nf, Co, Ci, x, x, None)
    out.append((n_, f_, 4 * L * S * (Ci + 2 * Co), 2.0 * Co * Ci * L * S))

    def reset():
        for t in st:
            t.zero_()
    return out, reset, keep


# NOTE on `algorithmic_bytes`: every figure follows SURVEY.md section 8(d) (each level's input read and output written
# once, merge reading every level), also for the one-pass pyramid, which really moves fewer bytes (y + z_0 + R_d once):
# its `frac` can therefore exceed what a level-by-level schedule could reach at the copy peak.


def time_block(w, B, stream, flush, dev, reps=7):
    """Times every kernel of one U-ConvBlock alone (L2 flushed before each launch) and the block as a whole
    (its kernels back to back as in the forward, L2 flushed before the block only).  CUDA events on the
    launching stream; medians."""
    peak, peak_src = load_peaks()
    am = algorithmic_model(w)
    launchers, reset, keep = block_launchers(w, B, dev, stream)

    def med(fn, n=reps):
        ms = []
        for _ in range(n):
            reset()
            flush.fill_(3)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            fn()
            e.record(stream)
            stream.synchronize()
            ms.append(s.elapsed_time(e))
        ms.sort()
        return ms[len(ms) // 2]

    def whole():
        for _, fn, _, _ in launchers:
            fn()
    for _ in range(2):
        reset()
        whole()
    stream.synchronize()
    kernels = []
    tpeak, tpeak_src = load_tensor_peak()
    for name, fn, nbytes, flops in launchers:
        t = med(fn)
        k = {"kernel": name, "avg_launch_ms": t, "algorithmic_bytes_per_launch": nbytes,
             "achieved": nbytes / t / 1e6, "frac": nbytes / t / 1e6 / peak,
             "tflops_fp32_equivalent": flops / t / 1e9}
        if "tcgen05" in name:       # fp32-grade result from 3 bf16 products per MAC: the tensor pipe sees 3x the flops
            k["bf16_tflops_issued"] = 3.0 * flops / t / 1e9
            k["frac_tensor"] = 3.0 * flops / t / 1e9 / tpeak
            k["tensor_peak_tflops"] = tpeak
            k["tensor_peak_source"] = tpeak_src
        kernels.append(k)
    t_blk = med(whole)
    gc = w["variant"] == "groupcomm"
    blk_bytes = B * (am["a_blk"] - (4 * am["L"] * 4 * w["kw"]["out_channels"] if gc else 0))   # TAC is not in this sequence
    per_block = {"ms": t_blk, "sum_of_kernels_ms": sum(k["avg_launch_ms"] for k in kernels),
                 "algorithmic_bytes": blk_bytes, "achieved": blk_bytes / t_blk / 1e6, "peak": peak, "unit": "GB/s",
                 "frac": blk_bytes / t_blk / 1e6 / peak,
                 "what": ("proj_1x1 -> causal depthwise stage -> res_conv+skip" if w["variant"] == "causal" else
                          "proj_1x1 -> depthwise levels -> merge -> res_conv+skip") + " of one U-ConvBlock at the benchmark "
                         "shape, launched back to back through the stage-level C-ABI (L2 flushed before the block)"}
    del keep
    return kernels, per_block, peak, peak_src


def roofline_block(w, B, stream, flush, dev):
    """`roofline` = the kernel with the largest share of the step (chosen from the measured per-kernel times, not
    assumed), next to every other kernel of the U-ConvBlock and the per-U-ConvBlock figure the north star names."""
    kernels, per_block, peak, peak_src = time_block(w, B, stream, flush, dev)
    top = max(kernels, key=lambda k: k["avg_launch_ms"])
    traffic = None      # dram__bytes_read+write per launch of that kernel at this shape, from the committed ncu capture
    tpath = os.path.join(REPO, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        for ent in (t if isinstance(t, list) else [t]):
            if ent.get("kernel_prefix") and top["kernel"].startswith(ent["kernel_prefix"]) and \
                    ent.get("algorithmic_bytes_per_launch") == top["algorithmic_bytes_per_launch"]:
                traffic = ent.get("dram_bytes_per_launch")
    return {"kernel": top["kernel"], "bound": "hbm", "achieved": top["achieved"], "peak": peak, "unit": "GB/s",
            "frac": top["frac"], "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": top["algorithmic_bytes_per_launch"], "avg_launch_ms": top["avg_launch_ms"],
            "selection": "largest measured per-launch time among the U-ConvBlock's kernels (16 launches of each per step)",
            "kernels": kernels, "per_block": per_block}


# --------------------------------------------------------------------------
# comparators next to the headline
# --------------------------------------------------------------------------
def eager_cuda_rate(w, B, dev, steps=5, warmup=2):
    """The reference's op sequence run by stock PyTorch eager kernels (ATen / cuDNN / cuBLAS) on this GPU: the
    oracle port on `cuda` (improved_sudormrf.py:283-301 under the notebook's timing protocol, :125-146).  This is the
    "existing Blackwell path" a user of the reference gets today; fp32, TF32 state recorded."""
    from oracle import sudormrf_oracle as O
    cfg = O.Config(variant=w["variant"], **w["kw"])
    sd = {k: v.to(dev) for k, v in O.make_state_dict(cfg, seed=0, perturbed=False).items()}
    x = torch.rand(B, 1, w["T"], generator=torch.Generator().manual_seed(1)).to(dev)
    ms = []
    with torch.no_grad():
        for _ in range(warmup):
            O.forward(cfg, sd, x)
        torch.cuda.synchronize(dev)
        for _ in range(steps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            O.forward(cfg, sd, x)
            e.record()
            torch.cuda.synchronize(dev)
            ms.append(s.elapsed_time(e))
    ms.sort()
    med = ms[len(ms) // 2]
    del sd, x
    torch.cuda.empty_cache()
    return {"value": B / (med / 1e3), "unit": UNIT, "ms_per_step": med, "batch": B, "steps": steps,
            "what": "oracle port of the reference forward executed by stock torch eager CUDA kernels on this GPU",
            "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
            "matmul_allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32), "dtype": "f32"}


def short_config_run(name, dev, stream, flush, steps=5, warmup=3):
    """A short device-resident run of another BASELINE config on this rank (same protocol as the headline)."""
    import sudo_rm_rf_b200 as P
    from oracle import sudormrf_oracle as O
    w = WORKLOADS[name]
    model = model_class(w["variant"])(**w["kw"])
    model.load_state_dict(O.make_state_dict(O.Config(variant=w["variant"], **w["kw"]), seed=0, perturbed=False))
    model = model.to(dev).eval()
    x = torch.rand(w["B"], 1, w["T"], generator=torch.Generator().manual_seed(7)).to(dev)
    with torch.no_grad(), torch.cuda.stream(stream):
        model(x)
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            model(x)
        for _ in range(warmup):
            graph.replay()
        stream.synchronize()
        tot = 0.0
        for _ in range(steps):
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            graph.replay()
            e.record(stream)
            stream.synchronize()
            tot += s.elapsed_time(e)
    n_params = sum(p.numel() for p in model.parameters())
    del graph, model, x
    torch.cuda.empty_cache()
    return w, tot / steps, n_params


def latency_b1(model, w, dev, stream, reps=20):
    """Batch-1 latency through the public host-buffer API (pinned in/out, CUDA-graph replay, sync per call):
    the protocol the reference publishes its GPU number with (B=1, notebook :125-146)."""
    hx = torch.rand(1, 1, w["T"]).pin_memory()
    hy = torch.empty(1, w["kw"]["num_sources"], w["T"]).pin_memory()
    with torch.no_grad(), torch.cuda.stream(stream):
        for _ in range(3):
            model.forward_host(hx, hy)
            stream.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            model.forward_host(hx, hy)
            stream.synchronize()
            ts.append(time.perf_counter() - t0)
    ts.sort()
    return {"ms": ts[len(ts) // 2] * 1e3, "best_ms": ts[0] * 1e3, "mixtures_per_s": 1.0 / ts[len(ts) // 2],
            "api": "model.forward_host, batch 1, host wall clock incl. H2D + D2H + sync", "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="improved_u16_512", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short runs of BASELINE configs 3 / 4 / 5")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's estimates as DIR/estimates.npy (float32; "
                         f"a seeded sample of batch rows above {DUMP_LIMIT_BYTES >> 20} MiB)")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w, args.workload)
    else:
        run_b200(args, w, args.workload)


if __name__ == "__main__":
    main()
