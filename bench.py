#!/usr/bin/env python
"""bench.py -- CTC-CRF loss+grad frames/sec on synthetic (N,T,V) log-probs (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (numerator + denominator forward-backward, loss and (N,T,V) gradient)
over one synthetic batch.  Workload at every N: the configuration the metric is quoted on --
N=64 utterances per GPU, T=1500, V=218, fp32, T-compose-LM den graph H=20000/d=24 (S=39999, A~1.02M arcs)
(SURVEY.md 8d).  Multi-GPU: every rank runs its own 64-utterance shard of a 64*N global batch (weak
scaling, no data-path collective) plus the path's single all-reduce of [sum cost, count].

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for how each field is obtained.
--dump-outputs DIR writes what the timed path returned in its last timed step (see dump_outputs) so that two builds can
be compared output for output: the inputs are seeded, identical from run to run for the same arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "CTC-CRF loss+grad frames/sec"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # workload overrides (development only; the defaults are the headline configuration)
    ap.add_argument("--N", type=int, default=64)
    ap.add_argument("--T", type=int, default=1500)
    ap.add_argument("--V", type=int, default=218)
    ap.add_argument("--H", type=int, default=20000)
    ap.add_argument("--d", type=int, default=24)
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--lamb", type=float, default=0.01)
    ap.add_argument("--varlen", action="store_true", help="variable-length batch (len ~ U{200..T}, sorted); not the headline workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--cpu-sample", default="auto", help="N,T of the CPU sample (default sized for ~15 s)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (global batches sharded over the ranks)")
    ap.add_argument("--strong-configs", default="5,4", help="which SURVEY configs the strong block runs (5: N=256 var-len; 4: N=128, 5M-arc graph)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss and gradient to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, sustained copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


_graph_dir = None


def den_graph_file(H, d, V):
    """The seeded synthetic den graph, written to a temporary directory of this process (removed at exit): the
    tree may be read-only, and a fixed name in a shared /tmp could be another user's or another version's file."""
    global _graph_dir
    from cat_b200 import fst
    if _graph_dir is None:
        _graph_dir = tempfile.TemporaryDirectory(prefix="ccb_bench_")
    path = os.path.join(_graph_dir.name, f"den_H{H}_d{d}_V{V}.fst")
    g = fst.make_synthetic_den(H, d, V, seed=7)
    if not os.path.exists(path):
        fst.write_fst(path, g)
    return path, g


DUMP_BYTES = 48_000_000     # what dump_outputs writes at most, headers aside


def dump_outputs(outdir, loss, grad):
    """What a caller of the timed path receives, as float32 or float64 .npy files: loss.npy, and the (N,T,V) gradient,
    as grad.npy when it fits DUMP_BYTES, otherwise as grad_rows.npy, the rows (n, t) of a fixed seeded sample, with
    grad_row_index.npy holding their indices n*T + t (the headline gradient is 84 MB)."""
    os.makedirs(outdir, exist_ok=True)
    grad = torch.as_tensor(grad)
    np.save(os.path.join(outdir, "loss.npy"), np.atleast_1d(torch.as_tensor(loss).detach().cpu().numpy()))
    if grad.numel() * grad.element_size() <= DUMP_BYTES:
        np.save(os.path.join(outdir, "grad.npy"), grad.detach().cpu().numpy())
        return
    rows = grad.detach().reshape(-1, grad.shape[-1])
    n_keep = DUMP_BYTES // (8 + rows.shape[1] * rows.element_size())
    idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], n_keep, replace=False))
    np.save(os.path.join(outdir, "grad_rows.npy"), rows[torch.from_numpy(idx).to(rows.device)].cpu().numpy())
    np.save(os.path.join(outdir, "grad_row_index.npy"), idx.astype(np.float64))


def synth_labels(N, T, V, seed, varlen=False):
    rng = np.random.default_rng(seed)
    lens = np.full(N, T, np.int32)
    if varlen:   # SURVEY 8d config 5: len ~ U{200..T}, sorted descending as sortedPadCollateASR does
        lens = np.sort(rng.integers(min(200, T), T + 1, size=N).astype(np.int32))[::-1].copy()
    ly = np.minimum(lens // 6, 400).astype(np.int32)
    labels = rng.integers(1, V, size=int(ly.sum())).astype(np.int32)
    return labels, lens, ly


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.skip = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            # nvidia-smi's own start-up (NVML init) stalls CUDA launches for tens of ms: let it finish BEFORE the
            # timed region starts, then drop what it printed while the GPU was idle
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:
                time.sleep(0.02)
            self.skip = len(self.rows)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.skip:]:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


CPU_SAMPLE_T = 32     # frames per utterance of the CPU legs' sample (the same in cpu_baseline and in --impl reference)


def cpu_port(graph, N, T, V, lamb, threads, seed=1234):
    """Times the fp64 oracle (oracle/ -- the CPU restatement; the reference has no CPU path) on a bounded
    sample of the workload.  Returns (frames/s, seconds, loss, grad)."""
    from oracle import oracle
    y, labels, lens, ly = oracle.synth_batch(N, T, V, seed=seed)
    t0 = time.perf_counter()
    loss, grad, _ = oracle.ctc_crf(graph, y, labels, lens, ly, lamb, True, nthreads=threads)
    dt = time.perf_counter() - t0
    return float(lens.sum()) / dt, dt, loss, grad


def run_reference(args, rank):
    """--impl reference: the reference path on the host cores.  The reference ships no CPU implementation
    (src/ctc_crf/setup.py:15-16), so this is the oracle port (kind "port"), all host threads, each step a
    bounded sample (N=cores, T<=64) of the same workload: same den graph, V, label density, lamb."""
    if rank != 0:
        return
    from oracle import oracle
    oracle.build()
    _, g = den_graph_file(args.H, args.d, args.V)
    cores = os.cpu_count() or 1
    sN = max(1, min(args.N, cores))
    sT = CPU_SAMPLE_T                 # the same T-slice as the cpu_baseline leg of the GPU arm
    cores = min(cores, sN)            # the port parallelises over utterances: threads actually used
    for _ in range(min(args.warmup, 1)):
        cpu_port(g, sN, sT, args.V, args.lamb, cores)
    t0 = time.perf_counter()
    frames = 0
    for k in range(args.steps):
        _, _, loss, grad = cpu_port(g, sN, sT, args.V, args.lamb, cores, seed=1234 + k)
        frames += sN * sT
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.float64(loss), grad)
    v = frames / dt
    sample = f"N={sN},T={sT} slice of the workload per step (same den graph, V, lamb)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"CTC-CRF loss+grad, N={args.N},T={args.T},V={args.V}, den S={g.num_states} A={g.num_arcs}",
                   "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "cpu_model": cpu_model(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    from cat_b200 import _C, _lib
    import ctc_crf

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    N, T, V = args.N, args.T, args.V
    path, graph = den_graph_file(args.H, args.d, V)
    ctx = ctc_crf.CRFContext(path, gpus=local_rank)
    info = _C.den_info()
    S_plan, A_file = info["states"], info["file_arcs"]     # algorithmic bytes use the den graph's own S and A (SURVEY 8d)
    dtype = torch.float32 if args.dtype == "f32" else torch.bfloat16
    b_in = 4 if args.dtype == "f32" else 2

    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    y = torch.log_softmax(3.0 * torch.randn(N, T, V, device=dev, generator=gen), -1).to(dtype).contiguous()
    labels_np, lens_np, ly_np = synth_labels(N, T, V, 1234 + rank, args.varlen)
    labels, lx, ly = torch.tensor(labels_np), torch.tensor(lens_np), torch.tensor(ly_np)
    frames_per_step = int(lens_np.sum())
    crit = ctc_crf.CTC_CRF_LOSS(lamb=args.lamb, size_average=True)

    host_s = [0.0, 0]   # host-side enqueue time of the resident steps (diagnostic: the GPU must never wait for it)
    last = {}           # the outputs of the latest resident step (--dump-outputs)

    def step_resident():
        t0 = time.perf_counter()
        loss, grad, _ = _C.ctc_crf_loss_fwd(y, labels, lx, ly, args.lamb, True)
        host_s[0] += time.perf_counter() - t0
        host_s[1] += 1
        if args.dump_outputs:
            last["loss"], last["grad"] = loss, grad
        if world > 1:
            v = torch.stack([loss.reshape(()) * N, torch.tensor(float(N), device=dev)])
            dist.all_reduce(v)
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        timed.launches_before = _C.launch_count()     # so that gpu_launches counts the timed steps only
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- value: whole-job throughput, inputs resident in HBM -------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("CCB_BENCH_NO_SAMPLER"):
        sampler.start()
    try:
        ms_total = timed(step_resident, args.steps, max(args.warmup, 3))
    finally:            # never leave nvidia-smi running behind
        clocks = sampler.stop() if rank == 0 else None
    launches = _C.launch_count() - timed.launches_before
    ms_per_step = ms_total / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["loss"], last["grad"])
    last.clear()
    value = world * frames_per_step / (ms_per_step * 1e-3)

    # ---- e2e: public API, host buffers, H2D of the step's logits + D2H of the loss inside the timed region ----
    y_host = y.cpu().pin_memory()
    y_dev = torch.empty_like(y)

    h2d_ev = []

    def step_e2e():
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        y_dev.copy_(y_host, non_blocking=True)
        eb.record()
        h2d_ev.append((ea, eb))
        loss = crit(y_dev.requires_grad_(False), labels, lx, ly)
        if world > 1:
            v = torch.stack([loss.reshape(()) * N, torch.tensor(float(N), device=dev)])
            dist.all_reduce(v)
        return float(loss.item())            # device->host read of the step's result

    e2e_steps = max(3, min(args.steps, 10))
    ms_e2e = timed(step_e2e, e2e_steps, 2) / e2e_steps
    e2e_value = world * frames_per_step / (ms_e2e * 1e-3)
    h2d_ms = sorted(a.elapsed_time(b) for a, b in h2d_ev[-e2e_steps:])   # the logits copy alone, per timed step
    meta_bytes = 4 * (labels.numel() + 3 * N + 1)
    h2d = y_host.numel() * y_host.element_size() + meta_bytes

    # ---- roofline: denominator forward-backward (the dominant kernels), timed live with CUDA events ----------
    L = _lib.lib()
    lens_dev = lx.to(dev)
    alpha_ws = torch.empty(int(L.ccb_den_alpha_floats(N, T)), dtype=torch.float32, device=dev)
    aux_ws = torch.empty(int(L.ccb_den_aux_bytes(N, T)), dtype=torch.uint8, device=dev)
    gden = torch.zeros(N, T, V, device=dev)
    logz = torch.empty(N, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    dcode = 0 if args.dtype == "f32" else 1

    def den(with_bwd):
        rc = L.ccb_den_forward_backward(y.data_ptr(), dcode, T * V, V, N, T, V, lens_dev.data_ptr(), alpha_ws.data_ptr(),
                                        aux_ws.data_ptr(), gden.data_ptr() if with_bwd else None, T * V, V, 1.0,
                                        logz.data_ptr(), None, stream)
        assert rc == 0, _lib.last_error()

    reps = max(2, min(args.steps, 5))
    ms_fwd = timed(lambda: den(False), reps, 1) / reps
    ms_fb = timed(lambda: den(True), reps, 1) / reps
    ms_bwd = max(ms_fb - ms_fwd, 1e-6)
    peak, peak_src = peaks()
    graph_bytes = A_file * 12 + S_plan * 16
    bytes_fwd = frames_per_step * (V * b_in + 4 * S_plan) + graph_bytes // 2
    bytes_bwd = frames_per_step * (V * b_in + 4 * V + 4 * S_plan) + graph_bytes // 2
    bytes_den = frames_per_step * (2 * V * b_in + 4 * V + 8 * S_plan) + graph_bytes
    ach = bytes_den / (ms_fb * 1e-3) / 1e9
    # measured DRAM traffic per launch: per-frame bytes from the committed ncu --set full capture (profiles/traffic.json,
    # taken at the same N/V/graph) x the frames of this launch; null for other workloads
    traffic = None
    pipes = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and (N, V, args.H, args.d, args.dtype) == (64, 218, 20000, 24, "f32"):
        tj = json.load(open(tpath))
        if "den_forward_kernel" in tj and "den_backward_kernel" in tj:
            traffic = (tj["den_forward_kernel"]["dram_bytes_per_frame"] + tj["den_backward_kernel"]["dram_bytes_per_frame"]) * T
            # instruction-pipe utilisation from the same committed ncu capture (BASELINE.md 3: report MUFU/FMA next to HBM)
            pipes = {k: {"fma": tj[k].get("pipe_fma_pct"), "xu": tj[k].get("pipe_xu_pct"), "issue_active": tj[k].get("issue_active_pct")}
                     for k in ("den_forward_kernel", "den_backward_kernel")}
            pipes["unit"] = "% of peak sustained active (ncu sm__inst_executed_pipe_*), " + tj["den_forward_kernel"].get("capture", "")
    roofline = {
        "bound": "hbm", "kernel": "den_forward_kernel + den_backward_kernel (denominator forward-backward)",
        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
        "traffic_ratio": (traffic / bytes_den) if traffic else None, "pipes": pipes, "peak_source": peak_src,
        "algorithmic_bytes": bytes_den,
        "algorithmic_bytes_per_frame": 2 * V * b_in + 4 * V + 8 * S_plan,
        "den_ms": ms_fb, "den_frames_per_s": frames_per_step / (ms_fb * 1e-3),
        "kernels": {
            "den_forward_kernel": {"ms": ms_fwd, "GB/s": bytes_fwd / (ms_fwd * 1e-3) / 1e9, "frac": bytes_fwd / (ms_fwd * 1e-3) / 1e9 / peak},
            "den_backward_kernel": {"ms": ms_bwd, "GB/s": bytes_bwd / (ms_bwd * 1e-3) / 1e9, "frac": bytes_bwd / (ms_bwd * 1e-3) / 1e9 / peak},
        },
        "arc_evals_per_s": 2.0 * A_file * frames_per_step / (ms_fb * 1e-3),
        "row_gathers_per_frame": info["fwd_slots"] + info["bwd_slots"],
        "l2_gather_TBps": (info["fwd_slots"] + info["bwd_slots"]) * T * (-(-N // (32 * (1 if N <= 32 else 2 if N <= 64 else 4)))) * (128 if N <= 32 else 256 if N <= 64 else 512) / (ms_fb * 1e-3) / 1e12,
    }
    del alpha_ws, aux_ws, gden

    # ---- strong scaling (SURVEY 8e, BASELINE configs 5 and 4): a FIXED global batch sharded over the ranks through
    # cat_b200.dist (length-balanced sharding, the CUDA op as the rank-local loss, ONE NCCL all-reduce of [sum cost, count]).
    # The same code runs at --gpus 1 (the whole batch on one GPU): speed-up at N GPUs = ms(1) / ms(N), taken from the
    # driver's back-to-back runs.  Each rank synthesises only its own shard (as a data loader would).
    def strong_case(tag, gN, gT, varlen, reps):
        from cat_b200 import dist as cdist
        labels_g, lens_g, ly_g = synth_labels(gN, gT, V, 4242, varlen)         # identical on every rank
        idx = cdist.shard_by_length(lens_g.tolist(), world)[rank]
        off = np.concatenate([[0], np.cumsum(ly_g)])
        lab_l = np.concatenate([labels_g[off[i]:off[i + 1]] for i in idx]) if idx else np.zeros(0, np.int32)
        lens_l, ly_l = lens_g[idx], ly_g[idx]
        Tl = int(lens_l.max()) if len(idx) else 1
        g2 = torch.Generator(device=dev).manual_seed(777 + rank)
        yl = torch.log_softmax(3.0 * torch.randn(len(idx), Tl, V, device=dev, generator=g2), -1).to(dtype).contiguous()
        shard = (idx, yl, torch.tensor(lab_l), torch.tensor(lens_l), torch.tensor(ly_l))
        loss_fn = cdist.cuda_loss_fn(args.lamb)
        last = {}

        def step():
            last["loss"], last["grad"] = cdist.sharded_step(loss_fn, shard, size_average=True)

        ms = timed(step, reps, 1) / reps
        frames = int(lens_g.sum())
        res = {"global_batch": gN, "max_len": int(lens_g.max()), "frames": frames, "ms_per_step": ms,
               "frames_per_s": frames / (ms * 1e-3), "local_utterances": len(idx), "local_frames": int(lens_l.sum()),
               "loss": float(last["loss"].item()), "reps": reps,
               "route": "cat_b200.dist.sharded_step(cuda_loss_fn): shard_by_length + fused CUDA loss per rank + 1 all-reduce of [cost,count]"}
        del yl, shard, last
        torch.cuda.empty_cache()
        return res

    strong = None
    strong_cfgs = [] if args.no_strong else [c.strip() for c in args.strong_configs.split(",") if c.strip()]
    if "5" in strong_cfgs and (N, V, args.H, args.d) == (64, 218, 20000, 24):
        strong = {"config5": dict(strong_case("config5", 256, 3000, True, 2),
                                  what="BASELINE config 5: N=256, len ~ U{200..3000} sorted, V=218, 1.02 M-arc den graph")}

    # ---- SURVEY 8f-1: raw-logit entry vs the caller's two-step path (log_softmax + loss + autograd), fwd+bwd ----
    raw_entry = None
    if world == 1:
        z = (3.0 * torch.randn(N, T, V, device=dev, generator=gen)).to(dtype)
        crit_raw = ctc_crf.CTC_CRF_LOSS(lamb=args.lamb, size_average=True, from_logits=True)

        def two_step():
            zz = z.detach().requires_grad_(True)
            crit(zz.float().log_softmax(-1), labels, lx, ly).backward()

        def fused():
            zz = z.detach().requires_grad_(True)
            crit_raw(zz, labels, lx, ly).backward()

        reps = max(2, min(args.steps, 5))
        ms_two, ms_fused = [], []
        for _ in range(2):   # alternate the two arms so that neither owns the warmer allocator / clocks
            ms_two.append(timed(two_step, reps, 2) / reps)
            ms_fused.append(timed(fused, reps, 2) / reps)
        raw_entry = {"two_step_ms": min(ms_two), "fused_ms": min(ms_fused), "all_ms": {"two_step": ms_two, "fused": ms_fused},
                     "what": "forward+backward from raw encoder outputs: torch log_softmax + CTC_CRF_LOSS + autograd vs CTC_CRF_LOSS(from_logits=True)"}
        del z

    if "4" in strong_cfgs and (N, V, args.H, args.d) == (64, 218, 20000, 24):
        del ctx
        path4, graph4 = den_graph_file(100000, 24, V)
        ctx = ctc_crf.CRFContext(path4, gpus=local_rank)       # the 5.09 M-arc graph replaces the 1.02 M-arc one on this device
        strong = strong or {}
        strong["config4"] = dict(strong_case("config4", 128, 2000, False, 1),
                                 what=f"BASELINE config 4: N=128, T=2000, V=218, den graph S={graph4.num_states} A={graph4.num_arcs}")
        del ctx
        ctx = ctc_crf.CRFContext(path, gpus=local_rank)

    out = None
    if rank == 0:
        # ---- reference CUDA build (B0) on the same GPU, and the CPU port on the host cores (N=1 run only) ----
        ref_cuda_res = None
        cpu_baseline = None
        if world == 1:
            if not args.no_ref_cuda:
                try:
                    from oracle import ref_cuda
                    if ref_cuda.available():
                        # BASELINE.md B0: the reference's CUDA code on this GPU.  At ~0.7 k frames/s the headline batch would
                        # take 140 s per repetition, so the arm runs the headline batch WIDTH (N utterances) over a T-slice
                        # (the reference launches 3T+6 kernels of N CTAs: its time per frame does not depend on T) --
                        # CUDA events on its stream, 1 warm-up + 3 timed repetitions, median.
                        rN, rT = N, min(T, 48)
                        rctx = ref_cuda.RefContext(path, local_rank)
                        yr = y[:rN, :rT].float().contiguous()
                        rlab, rlens, rly = synth_labels(rN, rT, V, 99)
                        args_ref = (rctx, yr, torch.tensor(rlab), torch.tensor(rlens), torch.tensor(rly), args.lamb, True)
                        ref_cuda.ctc_crf_forward(*args_ref)
                        torch.cuda.synchronize()
                        times = []
                        for _ in range(3):
                            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            ea.record()
                            ref_cuda.ctc_crf_forward(*args_ref)
                            eb.record()
                            torch.cuda.synchronize()
                            times.append(ea.elapsed_time(eb) * 1e-3)
                        rctx.close()
                        dt = sorted(times)[1]
                        ref_cuda_res = {"value": rN * rT / dt, "unit": UNIT, "reps_s": times,
                                        "sample": f"reference CUDA sources (oracle/_ref, sm_100a build with the two sm_100 fixes of oracle/Makefile) on this GPU, "
                                                  f"N={rN},T={rT} slice of the headline batch, same graph; CUDA events, 1 warm-up + 3 reps, median"}
                except Exception as e:  # the reference arm must never take the bench down
                    ref_cuda_res = {"error": repr(e)}
            if not args.no_cpu_baseline:
                from oracle import oracle
                oracle.build()
                cores = os.cpu_count() or 1
                if args.cpu_sample == "auto":
                    sN, sT = max(1, min(N, cores)), min(T, CPU_SAMPLE_T)
                else:
                    sN, sT = [int(x) for x in args.cpu_sample.split(",")]
                cores = min(cores, sN)    # the port parallelises over utterances: threads actually used
                v, dt, _, _ = cpu_port(graph, sN, sT, V, args.lamb, cores)
                cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "cpu_model": cpu_model(), "kind": "port", "seconds": dt,
                                "sample": f"fp64 oracle port (reference has no CPU path), N={sN},T={sT} slice, same den graph/V/lamb, {cores} threads"}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"CTC-CRF loss+grad N={N}/GPU,T={T},V={V} " + ("(variable lengths, SURVEY config 5 shape)" if args.varlen else "(BASELINE configs headline)"),
                       "den_graph": f"synthetic T-compose-LM H={args.H},d={args.d}: file S={graph.num_states} A={graph.num_arcs}; plan S={info['states']} pairs={info['pairs']} gathered arcs fwd/bwd={info['fwd_arcs']}/{info['bwd_arcs']}",
                       "global_batch": N * world, "parallelism": f"minibatch sharded x{world}, den graph replicated, 1 all-reduce of [cost,count]",
                       "lamb": args.lamb,
                       "l2": "no explicit flush: each step streams a 15.4 GB alpha spill (>> 126 MB L2)" if N * T >= 20000 else "small dev workload"},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                    "h2d_ms_median": h2d_ms[len(h2d_ms) // 2], "h2d_ms_max": h2d_ms[-1],
                    "api": "ctc_crf.CTC_CRF_LOSS.forward on pinned-host logits copied H2D inside the step, loss.item() back"},
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": 1e3 * host_s[0] / max(host_s[1], 1),
            "host_note": "host time inside the call; in the resident loop it is mostly the 4-slot pinned staging ring throttling the host to 4 steps ahead of the GPU (0.2 ms of real work per call, tools/host_probe.py)",
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "reference_cuda_same_gpu": ref_cuda_res,
            "raw_logit_entry": raw_entry,
            "strong": strong,
            "parity": {"vs_fp64_oracle": "loss 1e-4 relative, gradient 1e-3 absolute (occupancies in [0,1]) -- tests/test_gpu_atsize.py at this "
                                         "exact configuration and at BASELINE configs 1, 3, 4, 5, peaky logits and few final states",
                       "vs_reference_cuda": "loss 1e-4 relative, gradient 1e-3 at T=120 (tests/test_gpu_parity.py::test_vs_reference_cuda); at T >= 800 the "
                                            "reference's own fp32 log domain is 3.6e-2 away from the fp64 oracle (its occupancy rows do not sum to 1 "
                                            "within 3.6e-2), so the at-size bound is 'no farther from the oracle than the reference is' "
                                            "(test_full_size_properties)"},
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    del ctx
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
