#!/usr/bin/env python
"""bench.py — MSCKF + point-on-plane EKF updates/sec (BASELINE.json metric) on N B200s.

A "step" = one full UpdaterMSCKF::update-equivalent pass ("features triangulated, plane CPs known" -> posterior (x+, P+)) over the
synthetic workload BASELINE.json's metric is quoted on: N=512 state, 600 features (m=20) + 8 in-state planes
(`cfg3_n512_f600_p8`, SURVEY.md §8(d)): 8 sequential per-plane stacked updates + 1 point update.

  value : device-resident inputs (batch prepared once), per-step CUDA-event time on the library's stream, L2 flushed between steps
  e2e   : the same step through the C-ABI call with HOST buffers (plan + H2D + kernels + D2H of gates and state values), wall clock
  N > 1 : one independent filter replica per GPU (the per-plane update chain does not shard, DESIGN.md §multi-GPU), weak scaling;
          the sharded large-update path (cfg5: 4000 features, NCCL all-gather of compressed [R z] blocks) is reported beside it
  --impl reference : the reference's CPU algorithm (oracle restatement, the reference cannot be compiled here) on the host cores
  --dump-outputs DIR : the last `value` step's gates (feat_status, feat_chi2, plane_status, plane_chi2, hx_order) and posterior
          state (x: variable values in State::_variables order, P) as DIR/<name>.npy in float64, about 2 MB (rank 0);
          feat_chi2 / plane_chi2 hold only the individually gated features (feat_status 0, 1) / visited planes (plane_status 0, 1)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
WORKLOAD = "cfg3_n512_f600_p8"
METRIC = "MSCKF+plane EKF updates/sec at N=512 state, 600 feats"
UNIT = "updates/s"


def env_int(k, d):
    return int(os.environ.get(k, d))


class ClockSampler(object):
    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Rows that arrived inside [t0, t1] (the timed regions).  nvidia-smi is started BEFORE the warm-up, so it is already
        streaming when the timed region begins (started at the region's edge, its first row used to arrive after a 60 ms region
        had ended: zero samples)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.03)]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU algorithm (oracle restatement), all host cores = independent single-thread filters
# ------------------------------------------------------------------------------------------------------------------------
def _oracle_filter(job):
    """One single-thread reference filter pinned to one core: `warm` untimed + `steps` timed full updates of WORKLOAD (each from the
    same prior).  Returns per-step wall times, the reference's own per-stage timers and the gate counts."""
    seed, core, warm, steps = job
    if core is not None:
        try:
            os.sched_setaffinity(0, {core})
        except Exception:
            pass
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_backend  # bench.py may execute oracle/ only in the cpu_baseline and --impl reference legs
    from ov_plane_b200 import synth
    S = synth.make_scenario(WORKLOAD, seed=seed)
    chi2 = synth.chi2_table()
    times, stages, acc, planes = [], [], 0, 0
    for it in range(warm + steps):
        o = oracle_backend.OracleContext(S.options)
        o.set_chi2_table(chi2)
        ch = synth.load_scenario_into(o, S)
        b = synth.feature_batch(S, ch)
        t4 = np.zeros(4)
        t0 = time.perf_counter()
        r = o.msckf_update(b, 1.0, 1.0, timers=t4)
        dt = time.perf_counter() - t0
        o.close()
        if it >= warm:
            times.append(dt)
            stages.append(t4.tolist())
        acc, planes = int((r["feat_status"] == 1).sum()), int((r["plane_status"] == 1).sum())
    return times, stages, acc, planes, S.N, S.F


def workload_config(state_N, features, accepted, planes_passed):
    """The SAME object on the GPU line and on the reference line (the driver compares the two)."""
    return {"workload": WORKLOAD, "state_N": state_N, "features": features, "obs_per_feature": 20, "planes_in_state": 8,
            "accepted_point_features": accepted, "planes_passed": planes_passed,
            "parallelism": "replicas only (the per-plane update chain is sequential): one independent filter per GPU on the GPU arm, one "
                           "single-thread filter per pinned host core on the reference arm, N of them for --gpus N",
            "l2": "GPU arm: flushed between timed steps (256 MB write); reference arm: host caches, every step starts from a fresh state",
            "step": "restore(P, x) + 8 plane updates + 1 point update"}


def cpu_baseline_single():
    times, stages, acc, planes, N, F = _oracle_filter((0, None, 0, 1))
    dt, t4 = times[0], stages[0]
    return {"value": 1.0 / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "1 full %s update, single thread, oracle restatement of the reference's Givens/Eigen-order algorithm "
                      "(reference flags -O3, no Eigen available): %.2f s = plane updates %.2f + feature system %.2f + compression %.2f + "
                      "EKF update %.2f" % (WORKLOAD, dt, t4[0], t4[1], t4[2], t4[3])}


def run_reference(args):
    """The reference's update path is single-threaded (SURVEY.md fact 1).  Like the GPU arm (one filter replica per GPU, weak scaling),
    `--gpus N` runs exactly N concurrent single-thread filters, each pinned to its own core, each doing `warmup` untimed and `steps`
    timed full updates; value = sum over filters of 1 / median(step time).  If `steps` would not fit the time budget it is reduced
    and the line says so (`steps` is the number actually timed)."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    import multiprocessing as mp
    try:
        avail = sorted(os.sched_getaffinity(0))
    except Exception:
        avail = list(range(os.cpu_count() or 1))
    nf = max(1, min(args.gpus, len(avail)))
    cores = [avail[(i * len(avail)) // nf] for i in range(nf)]
    budget = 240.0
    # one untimed probe update on the first core sizes the run
    t_probe = _oracle_filter((0, cores[0], 0, 1))[0][0]
    warm = max(0, min(args.warmup, 1 if t_probe * (args.warmup + args.steps) > budget else args.warmup))
    steps = max(3, min(args.steps, int((budget - t_probe) / t_probe) - warm))
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(nf) as pool:
        res = pool.map(_oracle_filter, [(i, cores[i], warm, steps) for i in range(nf)])
    wall = time.perf_counter() - t0
    med = [float(np.median(r[0])) for r in res]
    allt = np.concatenate([np.asarray(r[0]) for r in res])
    value = float(sum(1.0 / m for m in med))
    st = np.median(np.concatenate([np.asarray(r[1]) for r in res]), axis=0)
    acc, planes, N, F = res[0][2], res[0][3], res[0][4], res[0][5]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * nf / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(N, F, acc, planes),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nf, "kind": "port",
                             "sample": "%d filter(s) x (%d warm-up + %d timed) full %s updates, oracle restatement of the reference's "
                                       "Givens/Eigen-order algorithm built with the reference's flags (no Eigen in this image); requested steps %d"
                                       % (nf, warm, steps, WORKLOAD, args.steps)},
            "step_seconds": {"median": float(np.median(allt)), "p95": float(np.percentile(allt, 95)), "min": float(allt.min()),
                             "max": float(allt.max()), "per_filter_median": med},
            "stage_seconds_median": {"plane_updates": float(st[0]), "feature_system": float(st[1]), "compression": float(st[2]),
                                     "ekf_update": float(st[3])},
            "host": {"cores_available": len(avail), "cores_used": cores, "wall_s": wall},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (gates and posterior x, P) "
                                                          "as DIR/<name>.npy, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from ov_plane_b200 import api, synth
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_over_ranks(x):
        if dist is None:
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    S = synth.make_scenario(WORKLOAD, seed=rank)
    chi2 = synth.chi2_table()
    ctx = api.Context(S.options, device=local, max_state=576, max_meas_rows=40000)
    ctx.set_chi2_table(chi2)
    ch = synth.load_scenario_into(ctx, S)
    batch = synth.feature_batch(S, ch)
    ctx.snapshot()
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def flush_l2():
        with torch.cuda.stream(stream):
            flush_buf.fill_(1.0)

    sampler = ClockSampler(local)
    sampler.start()
    # ---- warm-up through the full C-ABI path ----
    for _ in range(args.warmup):
        ctx.restore()
        out = ctx.msckf_update(batch, 1.0, 1.0)
    accepted = int((out["feat_status"] == 1).sum())
    planes_passed = int((out["plane_status"] == 1).sum())

    # ---- value: device-resident inputs, per-step CUDA events on the library's stream, L2 flushed between steps ----
    ctx.msckf_prepare(batch, 1.0, 1.0)
    ctx.restore()
    ctx.msckf_launch()
    ctx.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_region0 = time.time()
    l0 = ctx.launch_count()
    for k in range(args.steps):
        flush_l2()
        ev[k][0].record(stream)
        ctx.restore()
        ctx.msckf_launch()
        ev[k][1].record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    gates = ctx.msckf_finish()
    if args.dump_outputs:  # read back now: the passes below restore and update the same filter again
        # the ABI reports chi2 = NaN for features consumed by a plane update (status 2) and planes not visited (status -1):
        # keep the chi2 of the gated entries only, selected by status so that a NaN from a gated entry still shows
        gates["feat_chi2"] = gates["feat_chi2"][gates["feat_status"] != 2]
        gates["plane_chi2"] = gates["plane_chi2"][gates["plane_status"] != -1]
        dumped = {k: np.asarray(v, dtype=np.float64) for k, v in gates.items()}
        dumped["x"] = np.concatenate([ctx.var_get(h)[0] for h in ctx.variable_order()])
        dumped["P"] = ctx.cov()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    per_rank_ms = gather_over_ranks(float(np.mean(step_ms)))
    ms_per_step = max_over_ranks(float(np.mean(step_ms)))
    value = world / (ms_per_step * 1e-3)

    # ---- e2e: host buffers in, gates + state values out, every step ----
    h0, d0 = ctx.transfer_bytes()
    e2e_t = []
    barrier()
    for k in range(args.steps):
        flush_l2()
        ctx.restore()
        ctx.synchronize()
        t0 = time.perf_counter()
        out = ctx.msckf_update(batch, 1.0, 1.0)
        ctx.var_get(ctx.handle_imu())  # device->host read of the step's result (all variable values)
        e2e_t.append(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop(t_region0, time.time())  # nvidia-smi rows that arrived during the two timed regions (value + e2e)
    clocks["window"] = "device-timed steps + e2e steps"
    h1, d1 = ctx.transfer_bytes()
    n_var_bytes = 0
    e2e_ms = max_over_ranks(1e3 * float(np.mean(e2e_t)))
    sys.stderr.write("e2e per-step ms: %s\n" % " ".join("%.2f" % (1e3 * t) for t in e2e_t))
    e2e = {"value": world / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "ms_per_step_median": 1e3 * float(np.median(e2e_t)),
           "ms_per_step_max": 1e3 * float(np.max(e2e_t)),
           "h2d_bytes_per_step": int((h1 - h0) / args.steps), "d2h_bytes_per_step": int((d1 - d0) / args.steps) + n_var_bytes}

    # ---- roofline of the dominant kernel: per-kernel CUDA events on the launch stream (separate pass, not the timed region) ----
    ctx.msckf_prepare(batch, 1.0, 1.0)
    ctx.set_profiling(1)
    nprof = min(args.steps, 5)
    for _ in range(nprof):
        ctx.restore()
        ctx.msckf_launch()
    prof = ctx.profile_report()
    ctx.set_profiling(0)
    ctx.msckf_finish()
    peaks, peak_src = measured_peaks()
    # fp64 tensor peak is not in MEASURED_PEAKS.json: measure cuBLAS DGEMM here the way the driver measured bf16
    a = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
    b2 = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
    torch.matmul(a, b2)
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b2)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    fp64_peak = 2 * 4096 ** 3 / (best * 1e-3) / 1e12
    own_dgemm = ctx.selftest_dgemm_tflops(2048, 10)
    total_prof_ms = sum(v["ms"] for v in prof.values())
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
    dname, dv = dom
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(dname)
        except Exception:
            traffic = None
    if dname == "feature_kernel":
        ach = dv["work"] / (dv["ms"] * 1e-3) / 1e9
        roof = {"kernel": dname, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                "traffic": traffic, "peak_source": peak_src}
    else:
        ach = dv["work"] / (dv["ms"] * 1e-3) / 1e12
        roof = {"kernel": dname, "bound": "tensor", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                "traffic": traffic,
                "peak_source": "fp64: cuBLAS DGEMM 4096^3 via torch.matmul measured in this run (MEASURED_PEAKS.json has no fp64 entry; "
                               "its bf16 %.0f TF/s does not apply: the path computes in fp64 on DMMA, DESIGN.md)" % peaks.get("bf16_tflops", 0)}
    if dname == "chol_fused_kernel":
        roof["note"] = ("latency-bound: one cooperative launch factors a ~470-wide SPD system (and solves Y = M L^-T); the serial pivot chain, "
                        "not a throughput unit, bounds it (DESIGN.md 4.1) - frac against the tensor peak is reported as measured")
    roof["avg_launch_us"] = 1e3 * dv["ms"] / max(1, dv["launches"])
    roof["share_of_step"] = dv["ms"] / max(1e-9, total_prof_ms)
    roof["per_kernel_ms_per_step"] = {k: v["ms"] / nprof for k, v in prof.items()}
    roof["per_kernel_launches_per_step"] = {k: v["launches"] / nprof for k, v in prof.items()}
    roof["own_dgemm_tflops_2048"] = own_dgemm
    roof["algorithmic_flops_per_step"] = {k: v["work"] / nprof for k, v in prof.items() if k != "feature_kernel"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(S.N, S.F, accepted, planes_passed),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "per_rank_ms_per_step": per_rank_ms}

    # ---- throughput mode: C independent filters on ONE GPU, one stream + one CUDA graph each (the update chain of a single filter
    #      is latency-bound and occupies a few SMs at a time; independent filters fill the rest of the chip) ----
    try:
        C_f = 8
        others = []
        for i in range(C_f - 1):
            Si = synth.make_scenario(WORKLOAD, seed=100 + rank * 16 + i)
            ci = api.Context(Si.options, device=local, max_state=576, max_meas_rows=40000)
            ci.set_chi2_table(chi2)
            chi = synth.load_scenario_into(ci, Si)
            ci.snapshot()
            ci.msckf_prepare(synth.feature_batch(Si, chi), 1.0, 1.0)
            others.append(ci)
        ctx.msckf_prepare(batch, 1.0, 1.0)
        allc = [ctx] + others
        for _ in range(3):
            for ci in allc:
                ci.restore()
                ci.msckf_launch()
        for ci in allc:
            ci.synchronize()
        barrier()
        t0 = time.perf_counter()
        nrep = max(3, min(args.steps, 10))
        for _ in range(nrep):
            for ci in allc:
                ci.restore()
                ci.msckf_launch()
        for ci in allc:
            ci.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        for ci in allc:
            ci.msckf_finish()
        for ci in others:
            ci.close()
        agg = sum_over_ranks(C_f * nrep / dt)
        line["concurrent_filters"] = {"filters_per_gpu": C_f, "updates_per_s": agg, "ms_per_round": 1e3 * dt / nrep,
                                      "note": "independent filters on separate streams; same per-filter workload as `value`"}
    except Exception as e:
        line["concurrent_filters"] = {"error": repr(e)}

    # ---- propagation + clone as its own line (SURVEY 8(d)): Propagator::propagate_and_clone then marginalisation of the oldest
    #      clone (the per-frame pair that keeps N constant), same N = 512 state, 20 IMU samples per frame ----
    try:
        Sp = synth.make_scenario(WORKLOAD, seed=7)
        cp = api.Context(Sp.options, device=local, max_state=576, max_meas_rows=4096)
        cp.set_chi2_table(chi2)
        chp = list(synth.load_scenario_into(cp, Sp))
        cp.propagator_set_noise(1.6968e-04, 1.9393e-05, 2.0e-3, 3.0e-3, 9.81)
        tcur, dt_frame, nfr = Sp.timestamp, 0.05, 40
        rng = np.random.RandomState(1)
        for k in range(int((nfr + 2) * dt_frame / 0.0025) + 8):
            tt = tcur - 0.01 + 0.0025 * k
            cp.feed_imu(tt, np.array([0.05, -0.02, 0.1]) + 0.01 * rng.randn(3), np.array([0.1, 9.75, 0.3]) + 0.05 * rng.randn(3))
        for warm in (True, False):
            cp.synchronize()
            tw0 = time.perf_counter()
            for _ in range(4 if warm else nfr):
                tcur += dt_frame
                hnew = cp.propagate_and_clone(tcur)[0]
                cp.marginalize(chp.pop(0))
                chp.append(hnew)
            cp.synchronize()
            tw1 = time.perf_counter()
        line["propagation"] = {"ms_per_frame": 1e3 * (tw1 - tw0) / nfr, "frames_per_s": nfr / (tw1 - tw0), "state_N": cp.cov_rows(),
                               "imu_samples_per_frame": 20,
                               "note": "propagate_and_clone (host 15x15 IMU integration + EKFPropagation + augment_clone on the device) "
                                       "+ marginalize(oldest clone), wall clock through the C ABI"}
        cp.close()
    except Exception as e:
        line["propagation"] = {"error": repr(e)}

    # ---- BASELINE config 4: the ROS-free VioManager loop (30-clone window, room simulator) driving only the C ABI: propagate + clone,
    #      plane initialisation, MSCKF + plane update, marginalisation per camera frame (ov_plane_b200/vio_sim.py; parity: tests/test_gpu_vio.py) ----
    if rank == 0:
        try:
            from ov_plane_b200 import vio_sim
            o4 = vio_sim.state_options(max_clones=30)
            c4 = api.Context(o4, device=local, max_state=384, max_meas_rows=20000)
            c4.set_chi2_table(chi2)
            nfr4 = 120
            lp4, _ = vio_sim.run(c4, n_frames=nfr4, seed=3, max_clones=30)
            fr4 = lp4.frames[40:]
            est = np.array([r["propagation"] + r["plane_init"] + r["msckf"] + r["marg"] for r in fr4])
            line["cfg4"] = {"workload": "cfg4_room_sim_30clones (udel_room-like simulator, 60 tracked features, planes in the state)",
                            "frames": len(fr4), "state_N": int(fr4[-1]["N"]), "ms_per_frame_estimator": float(1e3 * est.mean()),
                            "ms_per_frame_estimator_p95": float(1e3 * np.percentile(est, 95)), "frames_per_s": float(1.0 / est.mean()),
                            "stage_ms": {k: float(1e3 * np.mean([r[k] for r in fr4])) for k in ("propagation", "plane_init", "msckf", "marg")},
                            "front_end_ms_python": float(1e3 * np.mean([r["front_end"] for r in fr4])),
                            "nees_ori": float(np.mean([r["nees_ori"] for r in fr4])), "nees_pos": float(np.mean([r["nees_pos"] for r in fr4])),
                            "final_err_deg_m": [float(fr4[-1]["err_ori_deg"]), float(fr4[-1]["err_pos"])],
                            "note": "wall clock of the estimator calls through the C ABI (the reference's timing-CSV columns, VioManager.cpp:911-928); "
                                    "simulator and Python front end excluded"}
            c4.close()
        except Exception as e:
            line["cfg4"] = {"error": repr(e)}

    # ---- PlaneFitting (SURVEY 8(f)3): RANSAC plane hypotheses + joint refinement for the 8 planes of the workload in one batch each ----
    if rank == 0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import planefit_cases
            ctx.restore()  # the clone poses the refinement problem was generated against
            fo8, pts8 = planefit_cases.plane_point_sets(S, seed=0)
            pr8 = planefit_cases.refine_problem(S, ch, seed=0, consistent=True, noise=0.006)
            fx8 = np.zeros(len(pr8["feat_offset"]) - 1, dtype=np.int32)
            tt = {"ransac": [], "refine": []}
            for it in range(8):
                ctx.synchronize()
                t0 = time.perf_counter()
                st8 = ctx.plane_fitting(fo8, pts8, 5, 200.0)[0]
                t1 = time.perf_counter()
                sr8 = ctx.optimize_plane(pr8["feat_offset"], pr8["meas_offset"], pr8["meas_clone"], pr8["uv_norm"], pr8["p_FinG"], pr8["cp_inG"], fx8,
                                         1.0 / 458.0, 0.01)
                t2 = time.perf_counter()
                if it >= 2:
                    tt["ransac"].append(t1 - t0)
                    tt["refine"].append(t2 - t1)
            line["plane_fit"] = {"planes": int(len(fo8) - 1), "points": int(fo8[-1]), "ransac_ms_per_batch": float(1e3 * np.mean(tt["ransac"])),
                                 "refine_ms_per_batch": float(1e3 * np.mean(tt["refine"])), "planes_fitted": int(st8.sum()),
                                 "refine_converged": int((sr8[4][:, 0] == 1).sum()), "refine_iterations": [int(x) for x in sr8[4][:, 1]],
                                 "note": "ovp_plane_fitting (200 hypotheses per plane, all planes concurrently) and ovp_optimize_plane (one launch: "
                                         "restated Ceres dogleg on per-feature blocks), host buffers in and out, wall clock"}
        except Exception as e:
            line["plane_fit"] = {"error": repr(e)}

    # ---- sharded large update (cfg5: 4000 features sharded over the ranks; the library owns the NCCL communicator and runs ONE
    #      all-gather of the packed rank-local Gram matrices inside ovp_msckf_update_sharded) - reported at N = 1 as well ----
    if not args.no_sharded:
        try:
            S5 = synth.make_scenario("cfg5_n512_f4000", seed=0)
            c5 = api.Context(S5.options, device=local, max_state=576, max_meas_rows=160000)
            c5.set_chi2_table(chi2)
            ch5 = synth.load_scenario_into(c5, S5)
            c5.snapshot()
            # rank 0 creates the communicator id; torch.distributed only carries the 128 bytes to the peers (plumbing)
            idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                idt.copy_(torch.frombuffer(bytearray(c5.nccl_unique_id()), dtype=torch.uint8))
            if dist is not None:
                dist.broadcast(idt, 0)
            c5.nccl_init(bytes(idt.cpu().numpy().tobytes()), world, rank)
            mine = [i for i in range(S5.F) if i % world == rank]
            b5 = synth.feature_batch(S5, ch5, mine)
            s5 = torch.cuda.ExternalStream(c5.stream(), device=torch.device("cuda", local))
            ts = []
            for it in range(3 + min(args.steps, 10)):
                c5.restore()
                barrier()
                t0 = torch.cuda.Event(enable_timing=True)
                t1 = torch.cuda.Event(enable_timing=True)
                t0.record(s5)
                c5.msckf_update_sharded(b5, ch5, 1.0, 1.0)
                t1.record(s5)
                barrier()
                if it >= 3:
                    ts.append(t0.elapsed_time(t1))
            sms = max_over_ranks(float(np.mean(ts)))
            n5 = c5.msckf_shard_columns(ch5)
            line["sharded_cfg5"] = {"workload": "cfg5_n512_f4000 (4000 features / %d ranks)" % world, "ms_per_update": sms, "updates_per_s": 1e3 / sms,
                                    "collective": "ncclAllGather of %d packed lower triangles of %d doubles, issued by the library on the ctx's own "
                                                  "communicator (ovp_msckf_update_sharded); summed in rank order, update replicated" %
                                                  (world, (n5 + 1) * (n5 + 2) // 2),
                                    "timing": "CUDA events on the library stream around the whole call (host plan + H2D + kernels + collective), "
                                              "max over ranks"}
            c5.nccl_finalize()
            c5.close()
        except Exception as e:  # the replica line above stays valid
            line["sharded_cfg5"] = {"error": repr(e)}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_single()
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in dumped.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
