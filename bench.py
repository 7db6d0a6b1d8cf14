#!/usr/bin/env python
"""bench.py -- headline benchmark of das4whales_b200 (contract: see the task statement).

Metric (BASELINE.json): DAS channels/s through the f-k filter (+ matched filter), plus achieved HBM GB/s vs the
measured roofline.  Workload at N=1: BASELINE.json configs[1] -- synthetic 10 000 ch x 120 000 samp fp32, f-k filter
only (dsp.fk_filter_design fan mask), 1 x B200.  At N>1 every rank filters its own 10 000 x 120 000 file (files are
independent: weak scaling, no data-path collective); additionally, at N>1, one 20 000 x 240 000 matrix is filtered
channel-sharded over all ranks with NCCL all-to-all transposes (BASELINE configs[3]) and reported under `sharded_fk`.

Extra legs in the same JSON line (all device-timed with CUDA events unless stated):
  hybrid_ninf               the mask every reference script uses (nothing prunable exactly) + its opt-in eps-pruned variant
  fk_plus_matched_filter    BASELINE configs[2]
  e2e                       dsp.fk_filter_filt with HOST buffers, H2D + D2H inside the timed region
  pipeline_e2e              BASELINE configs[4]'s per-GPU work: pipeline.MfDetectPipeline, int32 counts up, picks down
  cpu_baseline              the oracle port of the reference path on the box's host cores (N=1 only)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
"""
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

NX, NS = 10000, 120000
DX, FS = 2.0419046878814697, 200.0
FAN = (1400.0, 1450.0, 3400.0, 3500.0)
HYB = (1350., 1450., 3300, 3450, 14., 30.)      # scripts/main_mfdetect.py:46-47
ALGO_BYTES_PER_SAMPLE = 24          # SURVEY.md 8(d): 3 HBM round trips x (read + write) x 4 B
MF_BYTES_PER_SAMPLE = 12            # SURVEY.md 8(d): matched filter, 2 templates: read 4 + write 8
METRIC = "DAS channels/sec through f-k filter"
WORKLOAD = f"synthetic {NX} ch x {NS} samp fp32, f-k filter only (fk_filter_design fan mask {FAN}), one matrix per GPU"
CONFIG = {"workload": WORKLOAD, "l2": "inputs (4.8 GB) exceed the 126 MB L2; no flush needed"}   # identical in both arms
CPU_SAMPLE_NX = 250                 # single-thread sample: 250 channels x the full 120 000 samples
DUMP_ROWS, DUMP_SEED = 128, 0       # --dump-outputs: 128 full channels of the 4.8 GB output = 61 MB of float32
SHARD_NX, SHARD_NS = 20000, 240000  # BASELINE configs[3]

# ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per launch, keyed by what was profiled: (column scheme,
# kept rows).  Used only when the plan that runs equals the profiled one; otherwise `traffic` is null.
NCU_TRAFFIC = {(3, 1356): {"step": 7.390e9 + 2.547e9 + 3.256e9 + 2.546e9 + 8.044e9, "p5": 8.044e9,
                           "src": "profiles/r02_fk_pipe.txt (P1 7.390, P2 2.547, P3 3.256, P4 2.546, P5 8.044 GB)"}}
COL_KERNEL = {0: "k_col_inv_dual", 1: "k_col_inv_tma", 2: "k_colB_inv_fused + k_colA_inv", 3: "k_col2_pipe<inverse>"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def mem_available_gb():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 1048576.0
    except Exception:
        pass
    return 0.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def count_since(self, t_begin):
        return sum(1 for t, _ in self.rows if t >= t_begin)

    def stop(self, t_begin=0.0, window="timed region"):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if t < t_begin:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ---------------------------------------------------------------------------------------------------- CPU reference arm
def _cpu_inputs(nx):
    import numpy as np
    rng = np.random.default_rng(1234)
    return rng.standard_normal((nx, NS))


def _cpu_mask(nx):
    """fk_filter_design for an nx-channel sample, built in row chunks (oracle/torch_oracle.py, float64, CPU) so that the
    full 10 000 x 120 000 mask (9.6 GB) needs no 40 GB of temporaries."""
    from oracle import torch_oracle as TO
    return TO.fk_filter_design((nx, NS), [0, nx, 1], DX, FS, *FAN, device="cpu", rows_per_chunk=256).numpy()


_cpu_cache = {}


def time_cpu(nx, steps, warmup, workers):
    """oracle port of dsp.fk_filter_filt (dsp.py:725-756) on an nx-channel x 120 000-sample float64 matrix."""
    from oracle import dsp_oracle as O           # allowed here: cpu_baseline / --impl reference legs only
    if nx not in _cpu_cache:
        _cpu_cache.clear()
        _cpu_cache[nx] = (_cpu_inputs(nx), _cpu_mask(nx))
    x, mask = _cpu_cache[nx]
    fn = lambda: O.fk_filter_filt(x, mask, workers=workers)
    if workers is None and reference_source() == "reference":
        from oracle import ref_loader                # the unmodified reference function, where /root/reference is mounted
        ref_dsp = ref_loader.load()[0]
        fn = lambda: ref_dsp.fk_filter_filt(x, mask)
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        y = fn()
        dt = time.perf_counter() - t0
        del y
        if i >= warmup:
            ts.append(dt)
    t = sum(ts) / len(ts)
    return nx / t, t


def reference_source():
    """The unmodified reference is timed when /root/reference is mounted (build container); on the GPU box only the
    oracle port travels."""
    try:
        from oracle import ref_loader
        return "reference" if ref_loader.available() else "port"
    except Exception:
        return "port"


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    cores = len(os.sched_getaffinity(0)) or 1
    avail = mem_available_gb()
    full = avail >= 110.0 and os.environ.get("D4W_REF_FULL", "1") != "0"
    nx = NX if full else 1000
    # one untimed probe step sizes the run: the whole arm must end within a few minutes
    v0, t0 = time_cpu(nx, 1, 0, cores)
    eff_steps = max(1, min(steps, int(150.0 / max(t0, 1e-3))))
    eff_warm = 0 if t0 > 20 else min(warmup, 1)
    if eff_steps > 1 or eff_warm:
        val, t = time_cpu(nx, eff_steps, eff_warm, cores)
    else:
        val, t = v0, t0
    single, t1 = time_cpu(CPU_SAMPLE_NX, 1, 0, None)
    sample = (f"{nx} ch x {NS} samp float64 per step" + (" = the full workload matrix" if full else
              f" (1/{NX // nx} of the workload's channels, full time axis; host MemAvailable {avail:.0f} GB < 110 GB)"))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "channels/s", "n_gpus": args.gpus,
            "steps": eff_steps, "warmup": eff_warm, "requested_steps": steps, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": dict(CONFIG),
            "note": "reference CPU path = oracle port of dsp.fk_filter_filt (fft2 -> mask -> ifft2, complex128) with the FFTs on "
                    f"all {cores} host threads (scipy.fft, same pocketfft as numpy.fft); steps capped so that the arm ends in minutes; "
                    "the reference itself is single-threaded: see cpu_baseline.single_thread",
            "cpu_baseline": {"value": val, "unit": "channels/s", "cores": cores, "kind": "port", "sample": sample,
                             "full_matrix": full, "host_mem_available_gb": round(avail, 1),
                             "single_thread": {"value": single, "unit": "channels/s", "cores": 1,
                                               "kind": reference_source(),
                                               "sample": f"{CPU_SAMPLE_NX} ch x {NS} samp, numpy.fft exactly as the reference calls it"}},
            "e2e": {"value": val, "unit": "channels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------- host placement
def bind_to_gpu_numa(local):
    """Run this rank (and therefore first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs off."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node_path = f"/sys/bus/pci/devices/{bus}/numa_node"
        with open(node_path) as f:
            node = int(f.read().strip())
        if node < 0:
            return {"numa_node": node, "bound": False}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "bound": True, "cpus": len(cpus)}
        return {"numa_node": node, "bound": False}
    except Exception as exc:       # noqa: BLE001
        return {"bound": False, "why": repr(exc)[:120]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-mf", action="store_true", help="skip the f-k + matched-filter (BASELINE configs[2]) leg")
    ap.add_argument("--no-hybrid", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the filtered matrix of the last step as DIR/fk_filter_filt.npy: "
                         f"float32, the {DUMP_ROWS} channels drawn by numpy.random.default_rng({DUMP_SEED}), in ascending order "
                         "(rank 0's matrix when --gpus > 1)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    orig_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local)
    import numpy as np
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(minutes=8))
    import das4whales_b200 as dw
    from das4whales_b200 import _lib, synth
    from das4whales_b200.fk import FkFilter

    steps, warmup = max(1, args.steps), max(3, args.warmup)
    L = _lib.lib()
    mask = dw.dsp.fk_filter_design((NX, NS), [0, NX, 1], DX, FS, *FAN)
    flt = FkFilter(mask)
    x = synth.synth_strain(NX, NS, seed=1234 + rank)
    y = torch.empty_like(x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    def time_loop(fn, n):
        """device time per call: n calls bracketed by barrier + synchronize, CUDA events on the launching stream"""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b) / n)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # nvidia-smi needs ~1 s to come up: start it before the warm-up
    for _ in range(warmup):
        flt(x, out=y)
    # ---- per-pass device times (CUDA events on the launching stream) -------------------
    names = ["p1_col_fwd", "p2_row_split", "p3_row_mid", "p4_row_unsplit", "p5_col_inv"]
    pass_ms = [0.0] * 5
    reps = 5
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(reps)]
    torch.cuda.synchronize()
    for r in range(reps):
        ev[r][0].record()
        for i in range(5):
            flt.run_pass(i + 1, x, y)
            ev[r][i + 1].record()
    torch.cuda.synchronize()
    for r in range(reps):
        for i in range(5):
            pass_ms[i] += ev[r][i].elapsed_time(ev[r][i + 1]) / reps

    # ---- the timed region: exactly K steps ------------------------------------------------
    n0 = L.d4w_launch_count()
    barrier()
    t_begin = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        flt(x, out=y)
    e1.record()
    barrier()
    launches = L.d4w_launch_count() - n0
    dump = None
    if args.dump_outputs and rank == 0:
        dump_rows = np.sort(np.random.default_rng(DUMP_SEED).choice(NX, size=DUMP_ROWS, replace=False))
        dump = y[torch.from_numpy(dump_rows).to(y.device)].cpu().numpy()
    clocks = None
    if rank == 0:
        # nvidia-smi reports every 100 ms; a short timed region (K steps of ~8 ms) may see fewer than three reports, so
        # the identical step keeps running, untimed, until three reports have been taken under the same load
        window = "timed region"
        t_cont = time.perf_counter()
        while sampler.proc and sampler.count_since(t_begin) < 3 and time.perf_counter() - t_cont < 3.0:
            for _ in range(8):
                flt(x, out=y)
            torch.cuda.synchronize()
            window = "timed region + untimed continuation of the same step (region shorter than 3 nvidia-smi periods)"
        clocks = sampler.stop(t_begin, window)
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / steps
    value = NX * world / (ms_step * 1e-3)
    peak, peak_src = measured_peak()

    # ---- the scripts' mask: hybrid_ninf (nothing exactly prunable) and its opt-in eps-pruned variant ------------------------
    hyb = None
    if not args.no_hybrid:
        hmask = dw.dsp.hybrid_ninf_filter_design((NX, NS), [0, NX, 1], DX, FS, *HYB)
        hsteps = min(steps, 8)
        hf_exact = FkFilter(hmask)
        hf_exact(x, out=y)
        ms_exact = time_loop(lambda: hf_exact(x, out=y), hsteps)
        y_exact = y.clone()
        rows_exact = hf_exact.rows_kept
        del hf_exact
        torch.cuda.empty_cache()
        eps = 1e-5
        hf_eps = FkFilter(hmask, eps=eps)
        hf_eps(x, out=y)
        ms_eps = time_loop(lambda: hf_eps(x, out=y), hsteps)
        d = (y.double() - y_exact.double())
        err_max = float(d.abs().max() / y_exact.abs().max())
        err_l2 = float(torch.linalg.vector_norm(d) / torch.linalg.vector_norm(y_exact.double()))
        del d, y_exact
        hyb = {"workload": f"same matrix, mask = hybrid_ninf_filter_design{HYB} (scripts/main_mfdetect.py:46-47)",
               "exact": {"value": NX * world / (ms_exact * 1e-3), "unit": "channels/s", "ms_per_step": ms_exact, "steps": hsteps,
                         "rows_kept": rows_exact, "roofline_frac": round(ALGO_BYTES_PER_SAMPLE * NX * NS / (ms_exact * 1e-3) / 1e9 / peak, 4)},
               "eps_pruned": {"eps": eps, "value": NX * world / (ms_eps * 1e-3), "unit": "channels/s", "ms_per_step": ms_eps,
                              "steps": hsteps, "rows_kept": hf_eps.rows_kept,
                              "roofline_frac": round(ALGO_BYTES_PER_SAMPLE * NX * NS / (ms_eps * 1e-3) / 1e9 / peak, 4),
                              "error_vs_exact": {"max_norm": err_max, "l2": err_l2},
                              "note": "opt-in (FkFilter(mask, eps=...) / d4w_fk_mask_prune): rows whose folded mask never exceeds eps "
                                      "are dropped; contract tolerance is 1e-4 max-norm"}}
        del hf_eps, hmask
        torch.cuda.empty_cache()

    # ---- BASELINE configs[2]: f-k filter + fin-whale matched filter (HF + LF templates, one pass over the filtered data)
    mf = None
    if not args.no_mf:
        tgrid = np.arange(NS) / FS
        tpls = [dw.detect.gen_template_fincall(tgrid, FS, 17.8, 28.8, 0.68), dw.detect.gen_template_fincall(tgrid, FS, 14.7, 21.8, 0.78)]

        def fk_mf():
            flt(x, out=y)
            outs = dw.detect.compute_cross_correlograms(y, tpls)
            del outs
        fk_mf()
        mf_steps = min(steps, 5)
        mf_ms = time_loop(fk_mf, mf_steps)
        mf_only = max(mf_ms - ms_step, 1e-6)
        alg = (ALGO_BYTES_PER_SAMPLE + MF_BYTES_PER_SAMPLE) * NX * NS
        mf = {"workload": "BASELINE configs[2]: the same matrix through the f-k filter, then detect.compute_cross_correlograms "
                          "with the HF (17.8-28.8 Hz, 0.68 s) and LF (14.7-21.8 Hz, 0.78 s) fin-whale templates",
              "value": NX * world / (mf_ms * 1e-3), "unit": "channels/s", "ms_per_step": mf_ms, "steps": mf_steps,
              "roofline": {"bound": "hbm", "algorithmic_bytes": alg, "achieved": round(alg / (mf_ms * 1e-3) / 1e9, 1), "peak": peak,
                           "unit": "GB/s", "frac": round(alg / (mf_ms * 1e-3) / 1e9 / peak, 4),
                           "matched_filter_alone": {"ms": round(mf_only, 3), "algorithmic_bytes": MF_BYTES_PER_SAMPLE * NX * NS,
                                                    "frac": round(MF_BYTES_PER_SAMPLE * NX * NS / (mf_only * 1e-3) / 1e9 / peak, 4),
                                                    "includes": "row statistics pass + overlap-save correlation kernel"}}}
        torch.cuda.empty_cache()

    # ---- end to end through the public API with HOST buffers ---------------------------------
    # A stream of files: every step copies that step's strain matrix from pinned host memory, filters it
    # through das4whales_b200.dsp.fk_filter_filt and copies the result back to pinned host memory.
    # Consecutive steps are software-pipelined over three CUDA streams (H2D of file i+1 and D2H of file
    # i-1 run under the filter of file i; PCIe is full duplex), double-buffered on the device.
    e2e = None
    pipe_e2e = None
    ok = 1
    hx = hy = None
    if not args.no_e2e:
        e2e_steps = min(steps, 6)
        try:                                   # 3 x 4.8 GB of pinned host memory per rank
            hx = torch.empty((NX, NS), dtype=torch.float32, pin_memory=True)
            hy = [torch.empty((NX, NS), dtype=torch.float32, pin_memory=True) for _ in range(2)]
        except Exception:                      # noqa: BLE001 -- report, never hang the other ranks
            ok = 0
        if world > 1:
            flag = torch.tensor([ok], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = int(flag.item())
    if not args.no_e2e and not ok:
        e2e = {"unavailable": "pinned host buffers could not be allocated on every rank"}
        hx = hy = None
    elif not args.no_e2e:
        hx.copy_(x)
        torch.cuda.synchronize()
        del y
        xd = [x, torch.empty_like(x)]
        s_h2d, s_d2h = torch.cuda.Stream(), torch.cuda.Stream()
        s_cmp = torch.cuda.current_stream()

        def run_pipeline(n):
            ev_in = [None, None]       # H2D of buffer b finished
            ev_use = [None, None]      # filter finished reading buffer b
            ev_out = [None, None]      # D2H into host buffer b finished
            outs = [None, None]
            for i in range(n):
                bsel = i % 2
                with torch.cuda.stream(s_h2d):
                    if ev_use[bsel] is not None:
                        s_h2d.wait_event(ev_use[bsel])
                    xd[bsel].copy_(hx, non_blocking=True)
                    ev_in[bsel] = torch.cuda.Event(); ev_in[bsel].record(s_h2d)
                s_cmp.wait_event(ev_in[bsel])
                out = dw.dsp.fk_filter_filt(xd[bsel], mask)            # the public call (tensor in -> tensor out)
                ev_use[bsel] = torch.cuda.Event(); ev_use[bsel].record(s_cmp)
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(ev_use[bsel])
                    if ev_out[bsel] is not None:
                        s_d2h.wait_event(ev_out[bsel])
                    hy[bsel].copy_(out, non_blocking=True)
                    out.record_stream(s_d2h)
                    ev_out[bsel] = torch.cuda.Event(); ev_out[bsel].record(s_d2h)
                outs[bsel] = out
            torch.cuda.synchronize()

        run_pipeline(2)                                              # warm-up (allocator, plans)
        barrier()
        t0 = time.perf_counter()
        run_pipeline(e2e_steps)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": NX * world * e2e_steps / dt, "unit": "channels/s", "h2d_bytes_per_step": NX * NS * 4,
               "d2h_bytes_per_step": NX * NS * 4, "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3,
               "api": "das4whales_b200.dsp.fk_filter_filt(cuda tensor, FkMask); per step: pinned-host H2D of the input matrix, "
                      "filter, D2H of the filtered matrix to pinned host memory; steps pipelined over 3 streams (wall clock "
                      "around all steps incl. the final synchronize)"}
        del hy, xd
        x = None
        torch.cuda.empty_cache()

        # ---- BASELINE configs[4] per-GPU work: the whole detection pipeline, raw int32 counts up, picks down ----------------
        if not args.no_pipeline:
            try:
                from das4whales_b200 import pipeline
                scale = 4.0838e-11 * 1550.0 / 2.0419
                hraw = hx.view(torch.int32)                               # re-use the pinned buffer for the raw counts
                xs = synth.synth_strain(NX, NS, seed=1234 + rank)
                hraw.copy_((xs * 5.0e4).round().to(torch.int32))
                del xs
                torch.cuda.empty_cache()
                pipe = pipeline.MfDetectPipeline(NX, NS, [0, NX, 1], DX, FS, scale)
                npk = 0
                for res in pipe.stream([hraw]):                          # warm-up: plans, tables, allocator
                    npk = res["picks_hf"].shape[1] + res["picks_lf"].shape[1]
                p_steps = min(steps, 5)
                barrier()
                d2h = 0
                t0 = None
                # steady state of the file stream: the clock starts when the first file's picks are back (its successor's H2D
                # is then already in flight) and stops after p_steps further files -- the one-off pipeline fill is excluded
                for k, res in enumerate(pipe.stream([hraw] * (p_steps + 1))):
                    if k == 0:
                        t0 = time.perf_counter()
                        continue
                    d2h += 4 * (NX + 1) * 2 + 4 * (res["picks_hf"].shape[1] + res["picks_lf"].shape[1])
                torch.cuda.synchronize()
                dt = max_over_ranks(time.perf_counter() - t0)
                barrier()
                pipe_e2e = {"workload": "BASELINE configs[4] per-GPU work: pipeline.MfDetectPipeline = raw2strain -> bp_filt(14-30 Hz) -> "
                                        "hybrid_ninf f-k filter -> HF + LF matched filter -> threshold -> envelope -> prominence picks "
                                        "(scripts/main_mfdetect.py:42-103); one 10 000 x 120 000 int32 file per step and GPU",
                            "value": NX * world * p_steps / dt, "unit": "channels/s", "ms_per_step": dt / p_steps * 1e3, "steps": p_steps,
                            "h2d_bytes_per_step": NX * NS * 4, "d2h_bytes_per_step": d2h // p_steps, "picks_per_file": npk,
                            "h2d_floor_ms_at_55GBs": round(NX * NS * 4 / 55e9 * 1e3, 1),
                            "timing": "wall clock over p_steps files in the steady state of pipe.stream (H2D of file i+1 under the "
                                      "processing of file i); the first file's exposed H2D (pipeline fill) is outside the clock"}
                del pipe
            except Exception as exc:        # noqa: BLE001
                pipe_e2e = {"unavailable": repr(exc)[:300]}
        del hx
        torch.cuda.empty_cache()

    # ---- BASELINE configs[3]: ONE 20 000 x 240 000 matrix channel-sharded over all ranks (N > 1 only) ---------------------------
    sharded = None
    if world > 1 and not args.no_sharded:
        x = y = None
        torch.cuda.empty_cache()
        try:
            from das4whales_b200 import dist as d4wdist
            smask = dw.dsp.fk_filter_design((SHARD_NX, SHARD_NS), [0, SHARD_NX, 1], DX, FS, *FAN)
            xl = synth.synth_strain(SHARD_NX // world, SHARD_NS, seed=99 + rank, calls_per_minute=0)
            # (1) serial schedule (one slab per rank, blocking exchanges) with per-stage device times
            be = d4wdist.CudaBackend(smask, SHARD_NX, SHARD_NS, world)
            sflt = d4wdist.ShardedFkFilter(SHARD_NX, SHARD_NS, be)
            sflt(xl)
            barrier()
            s_steps = min(steps, 4)
            serial_ms = time_loop(lambda: sflt(xl), s_steps)
            stage_ms = {}
            for _ in range(2):
                sflt(xl, timers=stage_ms)
            stage_ms = {k: round(v / 2, 3) for k, v in stage_ms.items()}
            a2a_ms = sum(v for k, v in stage_ms.items() if k.startswith("a2a"))
            rows_kept = be.rows
            del sflt, be
            torch.cuda.empty_cache()
            # (2) overlapped schedule: sub-slabs, asynchronous all-to-alls one sub-slab ahead of the column transforms
            nsub = d4wdist.pick_nsub(SHARD_NS, world)
            be = d4wdist.CudaBackend(smask, SHARD_NX, SHARD_NS, world, nsub=nsub)
            sflt = d4wdist.ShardedFkFilter(SHARD_NX, SHARD_NS, be)
            sflt(xl)
            barrier()
            sh_ms = time_loop(lambda: sflt(xl), s_steps)
            # exchange volume per rank and direction: two real-matrix transposes + two pruned-spectrum transposes
            cpr, slab = SHARD_NX // world, SHARD_NS // world
            real_b = cpr * slab * 4 * (world - 1)
            spec_b = (rows_kept // world) * slab * 8 * (world - 1)
            sharded = {"workload": f"BASELINE configs[3]: ONE {SHARD_NX} x {SHARD_NS} matrix, channel-sharded over {world} GPUs, f-k filter "
                                   "(fan mask) with 4 NCCL all-to-all transposes (das4whales_b200.dist.ShardedFkFilter)",
                       "value": SHARD_NX / (sh_ms * 1e-3), "unit": "channels/s", "ms_per_step": sh_ms, "steps": s_steps, "nsub": nsub,
                       "schedule": "time slab cut into nsub sub-slabs; asynchronous all_to_all_single issued one sub-slab ahead, so "
                                   "NVLink transfers run under the column transforms",
                       "rows_kept": rows_kept, "nvlink_bytes_sent_per_rank_per_step": 2 * real_b + 2 * spec_b,
                       "serial_schedule": {"ms_per_step": serial_ms, "stage_ms_rank0": stage_ms, "all_to_all_ms": round(a2a_ms, 3),
                                           "compute_and_permute_ms": round(sum(stage_ms.values()) - a2a_ms, 3),
                                           "nvlink_gbs_per_rank_during_exchanges": round((2 * real_b + 2 * spec_b) / max(a2a_ms, 1e-6) / 1e6, 1)},
                       "note": "SURVEY 8(d) bound for 4 GPUs: 2 x 3.6 GB per GPU per direction at 900 GB/s = 8 ms of pure exchange"}
            del sflt, be, xl, smask
        except Exception as exc:            # noqa: BLE001
            sharded = {"unavailable": repr(exc)[:300]}
        torch.cuda.empty_cache()

    if rank == 0:
        algo_bytes = ALGO_BYTES_PER_SAMPLE * NX * NS
        achieved = algo_bytes / (ms_step * 1e-3) / 1e9
        traffic = flt.traffic_bytes()
        scheme = flt.plan.col_scheme
        prof = NCU_TRAFFIC.get((scheme, flt.rows_kept))
        kernels = {n: {"ms": round(pass_ms[i], 4), "actual_bytes": traffic[n],
                       "actual_gbs": round(traffic[n] / (pass_ms[i] * 1e-3) / 1e9, 1) if pass_ms[i] > 0 else None}
                   for i, n in enumerate(names)}
        dom_ms = pass_ms[4]
        dom_alg = 8 * NX * NS          # SURVEY 8(d) K3: 4 B read + 4 B written per (channel, sample)
        dom = {"name": COL_KERNEL.get(scheme, "?") + " (P5, C2R over channels)", "ms": round(dom_ms, 4), "algorithmic_bytes": dom_alg,
               "achieved": round(dom_alg / (dom_ms * 1e-3) / 1e9, 1), "frac": round(dom_alg / (dom_ms * 1e-3) / 1e9 / peak, 4),
               "traffic": prof["p5"] if prof else None}
        line = {"metric": METRIC, "value": value, "unit": "channels/s", "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": dict(CONFIG),
                "plan": {"rows_kept": flt.rows_kept, "rows_total": NX // 2 + 1, "t1": flt.plan.t1, "t2": flt.plan.t2,
                         "col_tile_samples": flt.plan.tile, "col_scheme": scheme, "plan_bytes_per_step": sum(traffic.values())},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(achieved / peak, 4), "traffic": prof["step"] if prof else None,
                             "traffic_source": ("ncu --set full dram__bytes_read+write per launch, " + prof["src"]) if prof else
                                               "no ncu capture of this exact plan (scheme, kept rows): see plan.plan_bytes_per_step "
                                               "for the bytes the plan must move",
                             "dominant_kernel": dom, "peak_source": peak_src,
                             "scope": "whole f-k filter = 5 kernels per step; achieved = 24 B/(channel*sample) algorithmic bytes "
                                      "(SURVEY 8d) / step time; actual_bytes per kernel below are lower because wavenumber rows "
                                      "with an identically-zero folded mask are never stored",
                             "kernels": kernels},
                "clocks": clocks, "host": {"numa": numa, "cores": os.cpu_count(), "mem_available_gb": round(mem_available_gb(), 1)}}
        if e2e:
            line["e2e"] = e2e
        if pipe_e2e:
            line["pipeline_e2e"] = pipe_e2e
        if hyb:
            line["hybrid_ninf"] = hyb
        if mf:
            line["fk_plus_matched_filter"] = mf
        if sharded:
            line["sharded_fk"] = sharded
        if not args.no_cpu_baseline and world == 1:
            try:
                os.sched_setaffinity(0, orig_affinity)      # the CPU baseline may use every host core again
            except Exception:                               # noqa: BLE001
                pass
            cores = len(os.sched_getaffinity(0))
            cv, ct = time_cpu(1000, 1, 0, cores)
            sv, st = time_cpu(CPU_SAMPLE_NX, 1, 0, None)
            line["cpu_baseline"] = {"value": cv, "unit": "channels/s", "cores": cores, "kind": "port",
                                    "sample": f"1000 ch x {NS} samp float64, one fk_filter_filt call ({ct:.1f} s): oracle port of the "
                                              "reference path with scipy.fft on all host threads (`bench.py --impl reference` runs the "
                                              "full 10 000-channel matrix when host memory allows)",
                                    "single_thread": {"value": sv, "unit": "channels/s", "cores": 1,
                                                      "kind": reference_source(),
                                                      "sample": f"{CPU_SAMPLE_NX} ch x {NS} samp ({st:.1f} s), numpy.fft as the reference calls it"}}
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "fk_filter_filt.npy"), dump)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
