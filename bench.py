#!/usr/bin/env python
"""bench.py -- ADMM iterations/sec of the B200 engine on BASELINE config C2.

A "step" is one ADMM iteration (one pass of the hot loop, solver.jl:140-165) on
the random sparse QP n=50k, m=100k, 1% density (nnz(A)=5e7), Nonneg+Box cones,
CG reduced-KKT solver, scaling=0, fixed rho, EmptyAccelerator (BASELINE.md 2).

  value     iterations/s, problem resident in HBM, loop timed with CUDA events on
            the engine stream (max over ranks).
  e2e       same metric through the public C-ABI calls with HOST buffers:
            update_qb + warm_start (H2D) + solve (K iterations) + result D2H,
            wall-clocked around the calls.  The one-time model upload is the
            analogue of the reference's `setup!`, which its own metric
            (times.iter_time / iter) excludes as well; it is reported as setup_s.
  roofline  dominant kernel = the CSR SpMV t = rho.*(A u): algorithmic bytes
            (12 B/nnz + vectors, SURVEY.md 8d) / CUDA-event time per launch.
  cpu_baseline  the oracle port (oracle/cosmo_oracle.py) on this box's host cores (sparse products of
            the KKT operator on all OpenMP threads), bounded sample of the same workload, setup excluded.
  parity    the engine's operator variable w against the oracle's after the same iterations on the
            identical arrays at full size (bound 1e-8, SURVEY 8c-ii).

`--impl reference` times the oracle port for the same K steps / W warm-up (the reference itself cannot run
here: no Julia; it has no C sources to compile).

`--dump-outputs DIR` writes the x, s, mu and objective of the timed solve (after exactly --steps iterations from a cold
start) as float64 .npy files, 2 MB at the default size: the problem comes from --seed, so two builds run with the same
arguments can be compared output for output.
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

METRIC = "ADMM iterations/sec"
UNIT = "iter/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=50_000)
    ap.add_argument("--m", type=int, default=100_000)
    ap.add_argument("--density", type=float, default=0.01)
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--cpu-sample-iters", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed solve returned (x, s, mu, obj_val) as float64 DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the engine's outputs (--impl b200)")
    return a


def workload_config(a, extra=None):
    cfg = {"workload": "C2 random sparse QP n=%d m=%d density=%g (nnz(A)=%d), Nonnegatives(m/2)+Box(m/2), "
                       "CGIndirectKKTSolver, scaling=0, adaptive_rho=false, EmptyAccelerator, cold start"
                       % (a.n, a.m, a.density, int(round(a.density * a.m)) * a.n),
           "n": a.n, "m": a.m, "seed": a.seed, "l2": "inputs_larger_than_L2 (A + A' = 1.2 GB streamed per operator application)",
           "sharding": "rows of A / cones split across ranks, n-vectors replicated, one allreduce(sum) per operator application"}
    if extra:
        cfg.update(extra)
    return cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

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
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_iterations(P, q, A, b, sets, iters, warm, keep_w_at=None, budget_s=None):
    """Time `iters` ADMM iterations of the oracle port after `warm` >= 1 untimed ones (same settings as the engine).
    setup() (the reference's setup!, excluded from its own iter_time too) runs before the clock starts; the sparse
    products of the KKT operator run on the host threads (oracle/fast_matvec.py), everything else is the oracle as is.
    The thread count is calibrated in situ during extra warm-up iterations (a container's CPU quota, wake-up latencies
    and NUMA placement make a stand-alone product benchmark a poor predictor: measured 10x off on the GPU box).
    Returns (seconds, iterations, mean CG iterations, host threads, w after `keep_w_at` iterations from the cold start or None)."""
    from oracle import cosmo_oracle as O
    from oracle import fast_matvec as F
    from oracle.bridge import to_oracle_cones
    cones = to_oracle_cones(sets)
    warm = max(1, warm)
    cands = F.thread_candidates() if F._threads is None else []
    probe = len(cands)                      # one extra warm-up iteration per candidate thread count
    marks, kept, per_t = {}, {}, {}

    def cb(it, ws):
        marks[it] = time.perf_counter()
        if 1 <= it <= probe:                # iteration `it` ran with cands[it - 1] threads ... (set below for the next one)
            per_t[cands[it - 1]] = marks[it] - marks.get(it - 1, t_first[0])
        if it < probe:
            F.set_threads(cands[it])
        elif it == probe and probe:
            F.set_threads(min(per_t, key=per_t.get))
        if budget_s is not None and it == probe + warm and it >= 2:
            # bounded sample: cut the timed iterations so that the run ends inside the budget (disclosed in `sample`)
            per_iter = marks[it] - marks[it - 1]
            left = budget_s - (marks[it] - t_first[0])
            fit = max(1, int(left / max(per_iter, 1e-9)))
            if fit < iters:
                st.max_iter = probe + warm + fit
        if keep_w_at is not None and it == keep_w_at:       # absolute iteration count from the cold start
            kept["w"] = ws.w.copy()

    st = O.Settings(kkt_solver="cg", scaling=0, adaptive_rho=False, max_iter=probe + warm + iters, eps_abs=0.0, eps_rel=0.0,
                    check_termination=25, check_infeasibility=40)
    ws = O.Workspace(P, q, A, b, cones, st)
    ws.setup()
    if probe:
        F._threads = cands[0]               # keeps threaded() from running its stand-alone calibration
        F.load().oracle_spmv_set_threads(cands[0])
    F.threaded(ws)
    t_first = [time.perf_counter()]
    res = ws.optimize(iter_callback=cb)
    iters = st.max_iter - probe - warm
    dt = marks[probe + warm + iters] - marks[probe + warm]
    inner = res.kkt.inner_iterations
    return dt, iters, float(np.mean(inner)) if inner else 0.0, F.threads_in_use(), kept.get("w")


def host_cores():
    try:
        from oracle import fast_matvec as F
        return F.usable_cpus()       # affinity mask capped by the container's CPU quota
    except Exception:
        return os.cpu_count() or 1


def run_reference(a, rank, world):
    if rank != 0:
        return
    import cosmo_b200
    P, q, A, b, sets = cosmo_b200.problems.random_sparse_qp(a.n, a.m, a.density, a.seed)
    # Same K steps and W warm-up iterations as the engine arm.  One ADMM iteration of C2 is ~110 sparse products of
    # 5e7 nonzeros: ~0.5 s on the host threads of a GPU box; the budget guard below only bites on small hosts.
    iters, warm = max(1, a.steps), max(2, a.warmup)
    budget_s = float(os.environ.get("COSMO_B200_REF_BUDGET_S", "270"))
    t0 = time.perf_counter()
    dt, iters, cg, threads, _ = oracle_iterations(P, q, A, b, sets, iters, warm, budget_s=budget_s)
    probe_s = time.perf_counter() - t0
    capped = iters < max(1, a.steps)
    val = iters / dt
    sample = ("%d ADMM iterations after %d warm-up iterations (requested %d/%d%s), the reference loop restated in "
              "NumPy (oracle/cosmo_oracle.py) with the sparse products of the KKT operator on %d OpenMP threads "
              "(oracle/spmv_omp.c; thread count calibrated on this host); setup excluded like in the reference's iter_time" % (
                  iters, warm, a.steps, a.warmup, ", capped by the %.0f s budget" % budget_s if capped else "", threads))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": iters,
            "warmup": warm, "ms_per_step": 1e3 * dt / iters, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(a, {"cg_iters_per_admm_iter": cg}),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "host_cores_available": host_cores(), "probe_s": probe_s},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    a = parse_args()
    # NCCL prints its version banner on STDOUT at NCCL_DEBUG=VERSION and at WARN (the GPU boxes export VERSION): keep
    # stdout for the one JSON line.  An explicit INFO / TRACE is the caller's choice and stays.
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
        os.environ.pop("NCCL_DEBUG", None)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return

    import torch
    import cosmo_b200
    from cosmo_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # ---- problem (identical on every rank: same seed) ---------------------------------
    t0 = time.perf_counter()
    P, q, A, b, sets = cosmo_b200.problems.random_sparse_qp(a.n, a.m, a.density, a.seed)
    gen_s = time.perf_counter() - t0
    n, m = a.n, a.m
    settings = cosmo_b200.Settings(scaling=0, adaptive_rho=False, max_iter=a.steps, eps_abs=0.0, eps_rel=0.0)

    t0 = time.perf_counter()
    shard = sharding.make_shard(P, q, A, b, sets, rank, world)
    eng = sharding.create_engine(shard, settings, device=local_rank, dist=dist)
    setup_s = time.perf_counter() - t0
    m_loc = shard.A.shape[0]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # pinned host buffers for the e2e leg
    pin = lambda k: torch.empty(k, dtype=torch.float64).pin_memory().numpy()
    hq, hb = pin(n), pin(m_loc)
    hq[:] = shard.q; hb[:] = shard.b
    hx0, hs0, hmu0 = pin(n), pin(m_loc), pin(m_loc)
    hx0[:] = 0; hs0[:] = 0; hmu0[:] = 0
    ox, os_, omu = pin(n), pin(m_loc), pin(m_loc)

    def run(iters):
        st = cosmo_b200.Settings(scaling=0, adaptive_rho=False, max_iter=iters, eps_abs=0.0, eps_rel=0.0).to_struct()
        eng.update_settings(st)
        eng.reset()
        return eng.solve(ox, os_, omu)

    # ---- warm-up --------------------------------------------------------------------------
    barrier()
    if a.warmup > 0:
        run(max(a.warmup, 3))
    # ---- timed: device-resident ---------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    out = run(a.steps)
    barrier()
    dev_s = out.times["iter_time_device"]
    if out.iter != a.steps:
        raise SystemExit("the timed solve stopped after %d of %d iterations (%s)" % (out.iter, a.steps, out.status))
    # the arrays the timed solve handed back; the later legs reuse the same host buffers
    result = {"x": ox.copy(), "s": os_.copy(), "mu": omu.copy(), "obj_val": np.array(out.obj_val)}
    # ---- timed: end to end through the C ABI with host buffers ----------------------------------
    st = cosmo_b200.Settings(scaling=0, adaptive_rho=False, max_iter=a.steps, eps_abs=0.0, eps_rel=0.0).to_struct()
    eng.update_settings(st)
    eng.reset()
    barrier()
    t0 = time.perf_counter()
    eng.update_qb(hq, hb)
    eng.warm_start(hx0, hs0, hmu0)
    out2 = eng.solve(ox, os_, omu)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel (CUDA events on the engine stream) -------------------------
    ms_A, bytes_A = eng.spmv_bench(0, 20)
    ms_At, bytes_At = eng.spmv_bench(3, 20)

    # ---- the ResultTimes split (types.jl:26-41) of a short extra run with the device phase timers on; outside the timed
    # region (the timers add event records around every phase) -- reporting only, never fatal
    phases = None
    try:
        k_ph = max(3, min(10, a.steps))
        stp = cosmo_b200.Settings(scaling=0, adaptive_rho=False, max_iter=k_ph, eps_abs=0.0, eps_rel=0.0, verbose_timing=True).to_struct()
        eng.update_settings(stp)
        eng.reset()
        barrier()
        outp = eng.solve(ox, os_, omu)
        barrier()
        phases = {"iters": k_ph, "proj_ms_per_iter": 1e3 * outp.times["proj_time"] / k_ph,
                  "kkt_ms_per_iter": 1e3 * outp.times["kkt_time"] / k_ph,
                  "iter_ms_per_iter": 1e3 * outp.times["iter_time_device"] / k_ph,
                  "note": "rank 0, CUDA events around the projection and the KKT solve (verbose_timing)"}
    except Exception as exc:                                   # noqa: BLE001
        phases = {"error": str(exc)[:200]}

    if dist is not None:
        t = torch.tensor([dev_s, e2e_s, ms_A, ms_At], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_s, e2e_s, ms_A, ms_At = [float(v) for v in t.tolist()]
        tb = torch.tensor([bytes_A, bytes_At], dtype=torch.float64, device="cuda")
        dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        bytes_A_all, bytes_At_all = [float(v) for v in tb.tolist()]
    else:
        bytes_A_all, bytes_At_all = bytes_A, bytes_At

    if rank == 0:
        peaks, peak_src = None, "fallback (B200_PROFILING.md: 6650 GB/s)"
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peak, peak_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        except Exception:
            peak = 6650.0
        ach_A = bytes_A / (ms_A * 1e-3) / 1e9
        ach_At = bytes_At / (ms_At * 1e-3) / 1e9
        # dram__bytes_read + dram__bytes_write of this kernel from the committed `ncu --set full` capture of the same
        # single-GPU command (profiles/): meaningful only for the unsharded matrix, null otherwise
        traffic = None
        if world == 1 and (a.n, a.m, a.density) == (50_000, 100_000, 0.01):
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "spmv_traffic.json"))).get("dram_bytes_per_launch")
            except Exception:
                pass
        cg = out.kkt_inner_iterations / max(out.iter, 1)
        line = {"metric": METRIC, "value": a.steps / dev_s, "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": 1e3 * dev_s / a.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(a, {"cg_iters_per_admm_iter": cg, "setup_s": setup_s, "problem_gen_s": gen_s,
                                              "kkt_multiplications": out.kkt_multiplications}),
                "e2e": {"value": a.steps / e2e_s, "unit": UNIT,
                        "h2d_bytes_per_step": 8.0 * (n + m_loc + n + 2 * m_loc) / a.steps,
                        "d2h_bytes_per_step": 8.0 * (n + 2 * m_loc) / a.steps,
                        "note": "update_qb + warm_start + solve(K iterations) + result download, host pinned buffers; "
                                "model upload (setup!) excluded like in the reference's iter_time",
                        "with_setup": {"value": a.steps / (e2e_s + setup_s), "unit": UNIT, "setup_s": setup_s,
                                       "note": "time to solution of a cold model: engine creation (CSC->CSR, slabs, "
                                               "upload) + the K iterations"}},
                "gpu_launches": int(out.kernel_launches),
                "clocks": clocks,
                "phases": phases,
                "roofline": {"bound": "hbm", "kernel": "spmv_win_kernel<double,EpiScale> (t = rho.*(A u), x staged in smem by TMA bulk copy)",
                             "achieved": ach_A, "peak": peak, "unit": "GB/s", "frac": ach_A / peak,
                             "traffic": traffic, "peak_source": peak_src, "ms_per_launch": ms_A,
                             "algorithmic_bytes_per_launch": bytes_A,
                             "other": {"kernel": "spmv_kernel<P> + spmv_win_kernel<double,EpiKktOp> (c = A't + P u + sigma u, dot u'c)",
                                       "achieved": ach_At, "frac": ach_At / peak, "ms_per_launch": ms_At,
                                       "algorithmic_bytes_per_launch": bytes_At}}}
        if not a.no_cpu_baseline and world == 1:
            scale = (a.n * a.m * a.density) / 5e7
            it_cpu = a.cpu_sample_iters if scale > 0.2 else 50
            k_par = 1 + it_cpu                      # compare w after the oracle's warm-up + sampled iterations
            dt, iters, cgc, threads, w_ref = oracle_iterations(P, q, A, b, sets, it_cpu, 1, keep_w_at=k_par)
            line["cpu_baseline"] = {"value": iters / dt, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "%d ADMM iterations of the same workload after 1 warm-up iteration (setup "
                                              "excluded, %.1f CG its/iter), oracle port with the KKT operator's sparse "
                                              "products on %d OpenMP threads" % (iters, cgc, threads),
                                    "host_cores_available": host_cores()}
            # parity on the identical arrays at full size: operator variable w after the same number of iterations
            st = cosmo_b200.Settings(scaling=0, adaptive_rho=False, max_iter=k_par, eps_abs=0.0, eps_rel=0.0).to_struct()
            eng.update_settings(st)
            eng.reset()
            eng.warm_start(hx0, hs0, hmu0)
            eng.solve(ox, os_, omu)
            w_gpu = eng.w()
            rel = float(np.max(np.abs(w_gpu - w_ref)) / max(np.max(np.abs(w_ref)), 1e-300)) if w_ref is not None else None
            line["parity"] = {"what": "max |w_engine - w_oracle| / max |w_oracle| after %d ADMM iterations on the identical "
                                      "(P, q, A, b, K) at full size" % k_par,
                              "value": rel, "bound": 1e-8, "ok": bool(rel is not None and rel <= 1e-8)}
        print(json.dumps(line))
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, result, shard, m, dist)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(path, result, shard, m, dist):
    """Rank 0 writes `result` as float64 .npy files; each rank's s and mu hold only its own rows, so under sharding
    they are gathered into the full m-vectors first (x and obj_val are the same on every rank)."""
    if dist is not None:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, (shard.rows, result["s"], result["mu"]))
        for k, name in ((1, "s"), (2, "mu")):
            full = np.empty(m)
            for p in parts:
                full[p[0]] = p[k]
            result[name] = full
    if shard.rank == 0:
        os.makedirs(path, exist_ok=True)
        for name, v in result.items():
            np.save(os.path.join(path, name + ".npy"), np.asarray(v, dtype=np.float64))


if __name__ == "__main__":
    main()
