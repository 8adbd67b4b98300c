#!/usr/bin/env python
"""bench.py — computeControl Hz of the B200 MPPI engine (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus N --steps K --warmup W [--workload autorally|cartpole|double_integrator_tube]
    python bench.py --impl reference ...      # the reference's CPU step() loop (oracle port) on the host cores
    python bench.py --all-configs             # one JSON line per BASELINE config C2..C5 (the last line is the headline C4)
    python bench.py --dump-outputs DIR ...    # also save what the last timed solve returned, as DIR/<workload>_<array>.npy

A "step" is one optimisation iteration of Controller::computeControl (noise draw -> N x T rollout -> baseline /
exp-weights -> weighted control average) on synthetic inputs (SURVEY.md §8d). Default workload = the configuration the
north-star target is quoted on: Autorally NN dynamics + map cost, N=32768, T=100 (BASELINE.json configs[3]); rollouts
are sharded over the N GPUs with ONE NCCL all-gather per solve (strong scaling: total work fixed).

Reported numbers
  value     solves/s with the inputs resident: K solves enqueued back to back (x0 / U travel in the kernel parameter
            bank), one sync at the end, CUDA events on the launching stream, max over ranks.
  e2e       solves/s through the public C-ABI call mppib_solve with HOST buffers, one blocking call per solve: host
            inputs -> device, result -> host every step (what Controller::computeControl does).
  roofline  K1 (fused rollout kernel): algorithmic bytes (N_local*T*C*4, one read of the noise buffer) / its average
            duration from CUDA events in a separate pass of the same process with L2 flushed between K0 and K1.
  cpu_baseline  the oracle (CPU port of the reference's launchCPURolloutKernel + host weight code) on the host cores
            (persistent worker pool, one pinned thread per core).
  reference_gpu  the UNMODIFIED reference GPU build (oracle/_ref/libmppi_ref_gpu.so: the reference's VanillaMPPIController
            and kernels compiled for sm_100 with an Eigen stand-in, "reference kernels, shimmed host") timed on the same
            box for C2 / C4: computeControl Hz with steady_clock around the host call, best of a few rollout block shapes.
  parity_ok (N > 1) the sharded solve against a single-GPU solve of the same seed, checked inside the warm-up.
Each timed region is exactly `steps` solves and the per-solve mean is reported; pick `steps` so that a region covers
>= 100 ms of work, or the number measures launch overhead and clock noise as much as the solve. How many solves come
before the last timed one depends only on the arguments, so with the same arguments the outputs saved by --dump-outputs
are comparable run to run and build to build.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "computeControl_hz"
UNIT = "solves/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, device_index: int):
        super().__init__(daemon=True)
        self.idx, self.stop_flag, self.samples, self.reasons, self.max_mhz = device_index, False, [], set(), None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _traffic_from_profile(workload_name: str, info: dict):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of K1 from the committed `ncu --set full` capture of this
    command (profiles/r02_final_*_k1_kernels.csv, written by tools/run_final_r02.sh + tools/summarize_ncu.py) — used only when
    that capture is of the SAME launch (grid and block of this run), otherwise None: a stale profile must not speak for a
    changed kernel."""
    import csv
    tag = "autorally" if workload_name.startswith("autorally_nn_N32768_T100") else (
        "racer" if workload_name.startswith("racer_lstm_H4_colored_N65536_T150") else None)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", f"r02_final_{tag}_k1_kernels.csv")
    if tag is None or not os.path.exists(path):
        return None, None
    try:
        rows = list(csv.reader(open(path)))
        rec = dict(zip(rows[0], rows[1]))

        def mbytes(prefix):
            for k, v in rec.items():
                if k.startswith(prefix):
                    unit = k[k.index("[") + 1:k.index("]")].lower()
                    return float(v) * {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[unit]
            raise KeyError(prefix)
        if int(float(rec["launch__grid_size []"])) != info["grid"] or int(float(rec["launch__block_size []"])) != info["block"]:
            return None, None
        return mbytes("dram__bytes_read.sum") + mbytes("dram__bytes_write.sum"), os.path.relpath(path, os.path.dirname(path) + "/..")
    except Exception:  # an unreadable summary is the same as no summary
        return None, None


def _workload(args):
    from mppi_generic_b200 import workloads as W
    return W.by_name(args.workload, args.rollouts, args.timesteps)


def _k1_variant(w):
    """Which form of the Autorally network K1 ran with (engine.cu: default mma.sync, env / flag overrides)."""
    if type(w.dyn).__name__ != "NeuralNetModel":
        return {}
    if os.environ.get("MPPIB_NN_TENSOR"):
        return {"nn_form": "tcgen05 3xTF32, FP32 accumulate"}
    if os.environ.get("MPPIB_NN_FFMA2"):
        return {"nn_form": "FP32 FFMA2 from shared memory"}
    return {"nn_form": "mma.sync m16n8k16, FP16 hi/lo operands in three products, FP32 accumulate (FP32-equivalent: "
                       "4e-7 max error against FP64, tests/test_nn_mma_scheme.py); state, cost and reductions in FP32"}


def _oracle_prepare(w):
    """The LSTM model's weights / architecture are handed to the oracle once (oracle/binding.py: set_lstm)."""
    import oracle
    if hasattr(w.dyn, "lstm_theta"):
        oracle.set_lstm(w.dyn.lstm_theta, w.dyn.hidden_dim, w.dyn.head_hidden)


def _cpu_solve_hz(w, nthreads, repeats, sample_N=None):
    """Times the oracle's full solve (setGaussianControls + CPU rollout + min/exp/sum + weighted reduction) on the host
    cores. Noise is pre-generated outside the timed region, as in the reference's CPU path, which reads the samples the
    GPU drew (tests/include/kernel_tests/core/rollout_kernel_test.cu:504-541). Returns (Hz of a FULL-size solve, text)."""
    import oracle
    _oracle_prepare(w)
    N = w.N if sample_N is None else min(sample_N, w.N)
    Cd = w.dyn.CONTROL_DIM
    eps = oracle.curand_normal(w.seed, 0, N * w.T * Cd).reshape(N, w.T, Cd)
    sp = w.sampler.params

    def once():
        return oracle.solve(w.dyn.DYN_ID, w.cost.COST_ID, w.dyn.params, w.cost.params, sp, w.dyn.nn_theta,
                            getattr(w.cost, "costmap", None), N, w.T, w.D, Cd, w.dt, w.lambda_, w.alpha, w.x0, w.U0, eps,
                            nthreads=nthreads)
    once()
    t0 = time.perf_counter()
    for _ in range(repeats):
        once()
    dt = (time.perf_counter() - t0) / repeats
    full = dt * (w.N / N)
    return 1.0 / full, f"{repeats} solves of {N}/{w.N} rollouts x {w.T} steps, {nthreads} threads, scaled to N={w.N}", dt


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path. The reference cannot be compiled here (all
    its host headers need Eigen, absent from this image; DESIGN.md), so this arm runs the oracle port of
    launchCPURolloutKernel + the host weight functions with all host threads, on the same workload/metric/unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = _workload(args)
    ncores = os.cpu_count() or 1
    # bound each step to roughly <= 1 s of CPU work: sample the rollouts if the full solve is longer
    hz_probe, _, dt_probe = _cpu_solve_hz(w, ncores, 1, sample_N=min(w.N, 2048))
    est_full = dt_probe * w.N / min(w.N, 2048)
    sample_N = w.N if est_full <= 1.5 else max(2048, int(w.N * 1.5 / est_full) // 64 * 64)
    import oracle
    N = min(sample_N, w.N)
    Cd = w.dyn.CONTROL_DIM
    eps = oracle.curand_normal(w.seed, 0, N * w.T * Cd).reshape(N, w.T, Cd)

    def once():
        oracle.solve(w.dyn.DYN_ID, w.cost.COST_ID, w.dyn.params, w.cost.params, w.sampler.params, w.dyn.nn_theta,
                     getattr(w.cost, "costmap", None), N, w.T, w.D, Cd, w.dt, w.lambda_, w.alpha, w.x0, w.U0, eps, nthreads=ncores)
    for _ in range(args.warmup):
        once()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        once()
    per = (time.perf_counter() - t0) / args.steps * (w.N / N)
    value = 1.0 / per
    sample = f"each step = CPU solve of {N}/{w.N} rollouts x {w.T} steps on {ncores} threads, scaled to N={w.N}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _base_config(w),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _dump_outputs(out_dir, w, U, stats):
    """What the last timed solve handed its caller: the optimal control sequence U [D][T][C] and, per distribution, the
    baseline (minimum sample cost), the normaliser (sum of the weights) and the sum of the squared weights."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"U": np.asarray(U, np.float32)}
    for i, key in enumerate(("baseline", "normalizer", "sum_w2")):
        arrays[key] = np.array([s[i] for s in stats], np.float32)
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, f"{w.name}_{key}.npy"), a)


def _base_config(w):
    """The keys both arms (--impl ours / reference) print under `config`, so that the driver's same-config check passes."""
    return {"workload": w.name, "num_rollouts": w.N, "num_timesteps": w.T, "controller": w.controller}


_REF_GPU_CHILD = r'''
import json, sys
sys.path.insert(0, sys.argv[3])
from mppi_generic_b200 import workloads as W
from oracle import ref_gpu as RG
name, b = sys.argv[1], tuple(int(v) for v in sys.argv[2].split(","))
w = W.by_name(name)
r = (RG.cartpole if name == "cartpole" else RG.autorally)(w, 42, block=b)
s = r.time_compute_control(w.x0[0], 1, warmup=5, iters=int(sys.argv[4]))
print("RESULT " + json.dumps({"block": list(b), "kernel": r.kernel_choice(), "ms": s * 1e3, "hz": 1.0 / s}))
'''
# rollout block shapes tried for the reference (dynamics x, y[, cost x, y]); the reference itself then picks its single or
# split rollout kernel by timing both. Each shape runs in its own process: the reference exit()s on a shape it rejects.
_REF_GPU_SHAPES = {"cartpole": ["64,4", "32,4", "64,1"], "autorally": ["64,8", "32,8", "64,4", "32,16"]}


def _reference_gpu(w):
    """computeControl Hz of the unmodified reference GPU build on this box (see the module docstring), or the reason it is
    not reported."""
    import subprocess
    from mppi_generic_b200 import workloads as W
    from oracle import ref_gpu as RG
    name = {"cartpole_vanilla_N8192_T100": "cartpole", "autorally_nn_N32768_T100": "autorally"}.get(w.name)
    if name is None:
        return {"unavailable": "the harness instantiates the reference for C2 (cartpole 8192 x 100) and C4 (autorally 32768 x 100) only"}
    if not RG.available():
        return {"unavailable": "oracle/_ref/libmppi_ref_gpu.so not built (oracle/ref_build/build.sh needs /root/reference)"}
    rows = []
    for b in _REF_GPU_SHAPES[name]:
        try:
            p = subprocess.run([sys.executable, "-c", _REF_GPU_CHILD, name, b, ROOT, "200" if name == "cartpole" else "40"],
                               capture_output=True, text=True, timeout=240)
            res = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
            rows.append(json.loads(res[0][7:]) if res else {"block": b, "error": (p.stdout + p.stderr)[-160:]})
        except Exception as ex:  # noqa: BLE001
            rows.append({"block": b, "error": str(ex)[:160]})
    ok = [r for r in rows if "hz" in r]
    if not ok:
        return {"unavailable": "every block shape failed", "tried": rows}
    best = max(ok, key=lambda r: r["hz"])
    return {"value": best["hz"], "unit": UNIT, "ms_per_call": best["ms"], "block": best["block"], "kernel": best["kernel"],
            "label": "reference kernels, shimmed host (unmodified /root/reference sources, Eigen stand-in, no-op feedback "
                     "controller), computeControl timed with steady_clock around the host call",
            "tried": rows}


def run_engine(args, ctx, emit=True, extra=None):
    """One workload through the engine; rank 0 prints the JSON line (emit) and returns it, the other ranks return None."""
    import torch
    import mppi_generic_b200 as m
    H = m.host
    dist, world, rank, local_rank = ctx

    w = _workload(args)
    # a real (non-default) stream: the legacy default stream has handle 0, which the C-ABI reads as "engine-owned", and
    # torch events would then not see the engine's work
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    flags = 0
    e = H.Engine(w.dyn, w.cost, w.sampler, w.N, w.T, w.D, device=local_rank, flags=flags,
                 stream=stream.cuda_stream, rank=rank, world_size=world)
    e.set_solver(w.dt, w.lambda_, w.alpha)
    e.seed(w.seed, 0)
    if world > 1:
        ids = [H.Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        e.comm_init(ids[0])
        if os.environ.get("MPPIB_NO_P2P") is None:
            e.p2p_setup(dist)  # peer-memory exchange on every rank, or NCCL on every rank

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    x0 = np.ascontiguousarray(w.x0, np.float32)
    U = np.ascontiguousarray(w.U0, np.float32).copy()
    U_out = np.empty_like(U)
    stats = (H.SolveStats * w.D)()

    # ---- multi-GPU parity, inside the warm-up: the sharded solve against a single-GPU solve of the same seed ------------
    parity = None
    if world > 1:
        e1 = H.Engine(w.dyn, w.cost, w.sampler, w.N, w.T, w.D, device=local_rank, flags=0, stream=stream.cuda_stream)
        e1.set_solver(w.dt, w.lambda_, w.alpha)
        e1.seed(w.seed, 0)
        U1, st1 = e1.solve(x0, U, w.optimization_stride, 0)
        e1.close()
        Us, sts = e.solve(x0, U, w.optimization_stride, 0)
        scale = max(1.0, float(np.abs(U1).max()))
        du = float(np.abs(Us - U1).max())
        ok = du <= 2e-5 * scale
        for d in range(w.D):
            ok = ok and sts[d][0] == st1[d][0] and abs(sts[d][1] - st1[d][1]) <= 1e-5 * abs(st1[d][1])
        t = torch.tensor([1.0 if ok else 0.0, du], device="cuda", dtype=torch.float64)
        dist.all_reduce(t[:1], op=dist.ReduceOp.MIN)
        dist.all_reduce(t[1:], op=dist.ReduceOp.MAX)
        parity = {"parity_ok": bool(t[0].item() == 1.0), "max_abs_dU_vs_single_gpu": float(t[1].item()),
                  "check": "sharded solve == single-GPU solve of the same seed: baseline identical, normaliser 1e-5, "
                           "U 2e-5 of the control scale, on every rank"}
        e.seed(w.seed, 0)

    # ---- warm-up, right before the timed solves (NVML start-up would otherwise leave the GPU idle in between) -------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        e.solve_into(x0, U, U_out, stats, w.optimization_stride, 0)
    n_timed = args.steps

    # ---- value: solves enqueued back to back, inputs resident (kernel parameter bank), device-timed ---------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(n_timed):
        e.solve_async(x0, U, w.optimization_stride, 0)
    ev1.record(stream)
    U_last, stats_last = e.solve_wait()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, w, U_last, stats_last)

    # ---- e2e: what Controller::computeControl does per call (mppi_controller.cu:151-241): one blocking C-ABI solve with
    # host buffers, then the host tail on the result — Savitzky-Golay smoothing and the nominal state/output roll-forward
    # (controller.cuh:557-663) through the library's host twins. Closed loop: the smoothed U feeds the next solve.
    Cd, S_, O_ = w.dyn.CONTROL_DIM, w.dyn.STATE_DIM, w.dyn.OUTPUT_DIM
    hist = np.zeros((2, Cd), np.float32)
    states = np.zeros((w.D, w.T, S_), np.float32)
    outputs = np.zeros((w.D, w.T, O_), np.float32)
    L = H.lib()

    # the host-tail calls with their ctypes arguments bound once (the C++ controller pays no marshalling at all; this
    # keeps the Python mirror's per-call overhead out of the number as far as ctypes allows)
    import ctypes as C
    tail_calls = []
    keep = []
    for d in range(w.D):
        up, sp_, op_ = U_out[d].ctypes.data, states[d].ctypes.data, outputs[d].ctypes.data
        tail_calls.append((L.mppib_host_smooth_controls, (up, hist.ctypes.data, w.T, Cd)))
        x0p = x0[d].ctypes.data
        if w.dyn.DYN_ID == H.DYN_RACER_LSTM:
            h0, c0 = w.dyn.initial_hidden_cell()
            net = w.dyn._host_net(h0, c0)
            keep += [h0, c0, net]
            tail_calls.append((L.mppib_host_output_trajectory_lstm,
                               (C.byref(w.dyn.params), C.byref(net), x0p, up, w.T, C.c_float(w.dt), sp_, op_)))
        else:
            nn = None if w.dyn.nn_theta is None else w.dyn.nn_theta.ctypes.data
            tail_calls.append((L.mppib_host_output_trajectory,
                               (w.dyn.DYN_ID, C.byref(w.dyn.params), nn, x0p, up, w.T, C.c_float(w.dt), sp_, op_)))

    def compute_control_separate():  # what the controller mirrors do: mppib_solve, then the host twins, call by call
        e.solve_into(x0, U, U_out, stats, w.optimization_stride, 0)
        for fn, a in tail_calls:
            fn(*a)
        U[...] = U_out

    cc_args = (e._h, x0.ctypes.data, U.ctypes.data, w.optimization_stride, 0, hist.ctypes.data, states.ctypes.data,
               outputs.ctypes.data, stats)
    is_user_pair = w.dyn.DYN_ID >= getattr(H, "USER_ID_BASE", 1 << 30)

    def compute_control():  # the same computeControl as ONE C-ABI call (mppib_compute_control), U updated in place
        if is_user_pair:
            return compute_control_separate()
        H._check(L.mppib_compute_control(*cc_args))

    for _ in range(3):
        compute_control()
    U[...] = w.U0
    barrier()
    ev0.record(stream)
    t0 = time.perf_counter()
    for _ in range(n_timed):
        compute_control()
    ev1.record(stream)
    torch.cuda.synchronize()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    e2e_ms = max(e2e_wall_ms, ev0.elapsed_time(ev1))
    # the same computeControl as separate calls (mppib_solve + host twins, what the header-only / Python controllers do)
    U[...] = w.U0
    t0 = time.perf_counter()
    for _ in range(n_timed):
        compute_control_separate()
    torch.cuda.synchronize()
    separate_ms = (time.perf_counter() - t0) * 1e3
    # the same loop without the host tail (C-ABI solve only), reported next to it
    U[...] = w.U0
    t0 = time.perf_counter()
    for _ in range(n_timed):
        e.solve_into(x0, U, U_out, stats, w.optimization_stride, 0)
        U[...] = U_out
    torch.cuda.synchronize()
    solve_only_ms = (time.perf_counter() - t0) * 1e3

    # the same computeControl with the tail ON THE DEVICE (SURVEY f2, mppib_nominal_trajectory chained behind the solve: one
    # host wait per call). Reported next to e2e; the host-twin tail above stays the default because it is faster.
    U[...] = w.U0
    U_s = np.empty_like(U)
    st_d = np.zeros((w.D, w.T, S_), np.float32)
    out_d = np.zeros((w.D, w.T, O_), np.float32)
    nt_args = (e._h, x0.ctypes.data, None, hist.ctypes.data, U_s.ctypes.data, st_d.ctypes.data, out_d.ctypes.data)
    device_tail_ms = None
    try:
        for it in range(3 + n_timed):
            if it == 3:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            e.solve_async(x0, U, w.optimization_stride, 0)
            H._check(L.mppib_nominal_trajectory(*nt_args))
            H._check(L.mppib_solve_wait(e._h, U_out.ctypes.data, stats))
            U[...] = U_s
        torch.cuda.synchronize()
        device_tail_ms = (time.perf_counter() - t0) * 1e3
    except H.MppibError as ex:  # a user pair without the call, Tsallis ...
        device_tail_ms = None
        print(f"[bench] device tail skipped: {ex}", file=sys.stderr)

    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.result()

    if dist is not None:
        t = torch.tensor([dev_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = float(t[0]), float(t[1])

    # ---- roofline pass: K1 duration from CUDA events, L2 flushed between K0 and K1, same process ----------------------
    U[...] = w.U0
    e.set_option(H.OPT_L2_FLUSH_BYTES, 256 << 20)
    e.enable_timing(True)
    for _ in range(max(10, min(args.steps, 50))):
        e.solve_into(x0, U, U_out, stats, w.optimization_stride, 0)
    t_cold = e.timing()
    e.set_option(H.OPT_L2_FLUSH_BYTES, 0)
    e.enable_timing(True)
    for _ in range(max(10, min(args.steps, 50))):
        e.solve_into(x0, U, U_out, stats, w.optimization_stride, 0)
    t_warm = e.timing()
    e.enable_timing(False)
    info = e.launch_info()
    peak, peak_src = _peaks()
    traffic, traffic_src = _traffic_from_profile(_base_config(w)["workload"], info) if world == 1 else (None, None)
    bytes_per_launch = e.n_local * w.T * w.dyn.CONTROL_DIM * 4
    achieved = bytes_per_launch / (t_cold["rollout_ms"] * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": "rollout kernel (K1)", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic,
        "traffic_note": ("dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of "
                         f"this command with the same grid / block ({traffic_src})") if traffic is not None else
                        "not measured in this run (no profiler attached) and no committed capture of this exact launch; the "
                        "ncu captures of this kernel are summarised under profiles/",
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": bytes_per_launch, "kernel_ms_l2_flushed": t_cold["rollout_ms"],
        "kernel_ms_l2_warm": t_warm["rollout_ms"],
        "stage_ms_l2_warm": {k: t_warm[k] for k in ("noise_ms", "rollout_ms", "reduce_ms", "total_ms")},
        "note": "K1 is bound by the T-step dependency chain (and MUFU / tensor-pipe work for NN dynamics), not by HBM: see DESIGN.md",
    }
    n_local = e.n_local
    e.close()
    line = None

    if rank == 0:
        value = n_timed / (dev_ms * 1e-3)
        e2e_value = n_timed / (e2e_ms * 1e-3)
        h2d = (x0.nbytes + U.nbytes)
        d2h = w.D * (w.T * w.dyn.CONTROL_DIM + 4) * 4
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            ncores = os.cpu_count() or 1
            hz, sample, _ = _cpu_solve_hz(w, ncores, 3, sample_N=None if w.N * w.T <= 4_000_000 else 8192)
            cpu = {"value": hz, "unit": UNIT, "cores": ncores, "kind": "port", "sample": sample}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / n_timed, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _base_config(w),
            "engine": {"parallelism": f"rollout-sharded dp{world}", "rollouts_per_gpu": n_local, "k1_launch": info,
                       "timed_solves": n_timed, "timed_ms": dev_ms,
                       **_k1_variant(w),
                       "l2": "noise buffer is regenerated on the device every solve (K0 -> K1 through L2/HBM); no data "
                             "is reused across solves; the roofline pass flushes L2 (256 MiB memset) between K0 and K1"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / n_timed,
                    "includes": "mppib_compute_control: blocking solve (host x0/U in, U/stats out) + host tail: SG smoothing and "
                                "nominal state/output roll-forward (T host step() calls), one C-ABI call per computeControl",
                    "separate_calls_value": n_timed / (separate_ms * 1e-3),
                    "solve_only_value": n_timed / (solve_only_ms * 1e-3),
                    "device_tail_value": None if device_tail_ms is None else n_timed / (device_tail_ms * 1e-3),
                    "device_tail_note": "same computeControl with smoothing + roll-forward as one device kernel chained "
                                        "behind the solve (mppib_nominal_trajectory); the host-twin tail is the default"},
            "gpu_launches": n_timed * info["kernels_per_solve"],
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if parity is not None:
            line.update(parity)
        if world == 1 and not args.no_reference_gpu:
            rg = _reference_gpu(w)
            line["reference_gpu"] = rg
            if "value" in rg:
                line["vs_reference_gpu"] = {"e2e_ratio": e2e_value / rg["value"], "value_ratio": value / rg["value"],
                                            "note": "north_star target: >= 10x the reference GPU build's computeControl Hz (C4)"}
        if extra:
            line.update(extra)
        if emit:
            print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
    return line if rank == 0 else None


def _setup():
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    return dist, world, rank, local_rank


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="autorally")
    ap.add_argument("--rollouts", type=int, default=None)
    ap.add_argument("--timesteps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed solve of each workload returned (U, baseline, normalizer, sum_w2) "
                         "as DIR/<workload>_<array>.npy")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="default run only: skip the C2 / C3 / C5 summaries carried in the headline line (other_configs)")
    ap.add_argument("--all-configs", action="store_true",
                    help="one JSON line per BASELINE config: C2 cartpole, C3 double_integrator_tube, C5 racer_lstm, then C4 "
                         "autorally (the headline, last)")
    args = ap.parse_args()
    workloads = ["cartpole", "double_integrator_tube", "racer_lstm", "autorally"] if args.all_configs else [args.workload]
    if args.impl == "reference":
        for wl in workloads:
            args.workload = wl
            run_reference(args)
        return
    ctx = _setup()
    extra = None
    if (not args.all_configs and args.workload == "autorally" and args.rollouts is None and args.timesteps is None
            and not args.no_other_configs):
        # the other BASELINE configs (C2, C3, C5), measured the same way in the same process and carried inside the
        # headline line as a summary, so that one default run shows every config at this GPU count
        import copy
        others = []
        for wl in ("cartpole", "double_integrator_tube", "racer_lstm"):
            sub = copy.copy(args)
            sub.workload, sub.no_cpu_baseline, sub.no_reference_gpu = wl, True, True
            ln = run_engine(sub, ctx, emit=False)
            if ln is not None:
                others.append({"workload": ln["config"]["workload"], "value": ln["value"], "unit": ln["unit"],
                               "e2e": ln["e2e"]["value"], "ms_per_step": ln["ms_per_step"],
                               "k1_ms_l2_flushed": ln["roofline"]["kernel_ms_l2_flushed"],
                               "k1_hbm_frac": ln["roofline"]["frac"], "stage_ms": ln["roofline"]["stage_ms_l2_warm"],
                               "timed_ms": ln["engine"]["timed_ms"], "parity_ok": ln.get("parity_ok")})
        extra = {"other_configs": others}
    for wl in workloads:
        args.workload = wl
        run_engine(args, ctx, extra=extra if wl == "autorally" else None)
    if ctx[0] is not None:
        ctx[0].destroy_process_group()


if __name__ == "__main__":
    main()
