#!/usr/bin/env python
"""bench.py -- Riccati knots/s of the B200 batched sweep (BASELINE.json metric).

One "step" = one backward(mueq)+forward() sweep (the loop body of the reference's
bench/gar-riccati.cpp:46-49) over a batch of synthetic LQ problems of BASELINE config 2
(nx=12, nu=6, nc=0, N=100, batch=4096 per GPU), all inputs resident in HBM.
  value     = batch*(N+1)*n_gpus / device time per step (CUDA events, max over ranks)
  e2e       = same metric through the C ABI with HOST (pinned) buffers: H2D of the knot
              records + sweep + D2H of gains and trajectories inside the timed region
  roofline  = algorithmic bytes per sweep (BASELINE.md section 3) / kernel time vs the
              measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline / --impl reference = the CPU oracle (restated reference algorithm, OpenMP
              over instances on all host cores) on a bounded sample of the same workload.
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

NX, NU, NC, NCT, HORIZON, BATCH = 12, 6, 0, 0, 100, 4096
MUEQ = 1e-11  # bench/gar-riccati.cpp:22
WORKLOAD = "batched synthetic LQR nx=12 nu=6 nc=0 N=100 batch=4096 per GPU (BASELINE config 2)"
# other BASELINE configs, selectable with --config for profiling (the default line is config 2)
CONFIGS = {
    "c2": (12, 6, 0, 0, 100, 4096, 1e-11, WORKLOAD),
    "c1": (6, 3, 0, 0, 100, 4096, 1e-11, "nx=6 nu=3 N=100 (BASELINE config 1 dims) batch=4096"),
    "c3": (4, 2, 2, 0, 100, 16384, 1e-3, "nx=4 nu=2 nc=2 N=100 batch=16384 (BASELINE config 3)"),
    "c4": (14, 7, 0, 0, 200, 2048, 1e-11, "nx=14 nu=7 N=200 batch=2048 (BASELINE config 4)"),
    "c5": (57, 28, 0, 0, 150, 512, 1e-11, "nx=57 nu=28 N=150 batch=512 (BASELINE config 5, CTA per instance)"),
}


def bytes_per_knot(nx, nu, nc):
    """BASELINE.md section 3: read knot + write ff,fb,Vxx,vx + write xs,us,vs,lbdas."""
    rd = 2 * nx * nx + 2 * nx * nu + nu * nu + 2 * nx + nu + nc * (nx + nu + 1)
    wr = (nu + nc + nx) * (nx + 1) + nx * nx + nx
    fw = 2 * nx + nu + nc
    return 8 * (rd + wr + fw)


def synth_batch_torch(torch, batch, N, nx, nu, device, seed, nc=0, nct=0, cstyle="control"):
    """SURVEY section 8(d) synthetic inputs (conditioned variant), generated on `device`,
    packed in the C-ABI layout [A|B|f|Q|S|R|q|r] (column-major blocks)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    f64 = torch.float64
    rn = lambda *s: torch.randn(*s, generator=g, device=device, dtype=f64)
    ru = lambda *s: torch.rand(*s, generator=g, device=device, dtype=f64) * 2 - 1
    n = nx + nu
    W = rn(batch, N, n, n + 1)
    H = W @ W.transpose(-1, -2) / max(nx, nu)
    Q, S, R = H[..., :nx, :nx], H[..., :nx, nx:], H[..., nx:, nx:].clone()
    R.diagonal(dim1=-2, dim2=-1).mul_(1 + 1e-6)
    A = torch.eye(nx, device=device, dtype=f64) + 0.1 * rn(batch, N, nx, nx) / nx ** 0.5
    Bm = ru(batch, N, nx, nu)
    cm = lambda M: M.transpose(-1, -2).reshape(batch, N, -1)  # column-major flatten
    parts = [cm(A), cm(Bm), rn(batch, N, nx), cm(Q), cm(S), cm(R), ru(batch, N, nx), ru(batch, N, nu)]
    if nc > 0 and cstyle == "control":  # C = 0, D = I rows with a random half zeroed (inactive box rows), d ~ U[-1,1]
        act = (torch.rand(batch, N, nc, generator=g, device=device, dtype=f64) < 0.5).to(f64)
        D = torch.eye(nc, nu, device=device, dtype=f64).expand(batch, N, nc, nu) * act[..., None]
        parts += [torch.zeros(batch, N, nc * nx, device=device, dtype=f64), cm(D), ru(batch, N, nc) * act]
    elif nc > 0:  # the reference generator's state constraints: C = I, D = 0, d ~ U[-1,1] (tests/gar/test_util.cpp:41-44)
        Cm = torch.eye(nc, nx, device=device, dtype=f64).expand(batch, N, nc, nx)
        parts += [cm(Cm), torch.zeros(batch, N, nc * nu, device=device, dtype=f64), ru(batch, N, nc)]
    stage = torch.cat(parts, dim=-1)
    if stage.shape[-1] % 2:
        stage = torch.cat([stage, torch.zeros(batch, N, 1, device=device, dtype=f64)], dim=-1)
    stage = stage.contiguous()
    Wt = rn(batch, nx, nx + 1)
    Qt = Wt @ Wt.transpose(-1, -2) / nx
    tparts = [Qt.transpose(-1, -2).reshape(batch, -1), ru(batch, nx)]
    if nct > 0:  # terminal knot: C = I (nct x nx), d ~ U[-1,1]
        Ct = torch.eye(nct, nx, device=device, dtype=f64).expand(batch, nct, nx)
        tparts += [Ct.transpose(-1, -2).reshape(batch, -1), ru(batch, nct)]
    term = torch.cat(tparts, dim=-1).contiguous()
    G0 = (-torch.eye(nx, device=device, dtype=f64)).expand(batch, nx, nx).reshape(batch, -1).contiguous()
    g0 = rn(batch, nx).contiguous()
    return stage, term, G0, g0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except ValueError:
                continue
            for nme, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(stage, term, G0, g0, nx, nu, nc, nct, N, target_s=12.0, max_inst=512):
    """Times the CPU oracle (OpenMP over instances, all host threads) on the first
    `max_inst` instances of the workload; repeats the sweep to reach ~target_s."""
    from oracle import gar_oracle as orc
    nb = min(max_inst, stage.shape[0])
    bo = orc.BatchedOracle(nx, nu, nc, nct, nx, N, nb, stage[:nb], term[:nb], G0[:nb], g0[:nb])
    threads = orc.num_threads()
    t1 = bo.sweep(MUEQ, reps=1)  # warm-up + calibration
    reps = max(1, min(200, int(target_s / max(t1, 1e-4))))
    t = bo.sweep(MUEQ, reps=reps)
    knots = nb * (N + 1) * reps
    return {"value": knots / t, "unit": "knots/s", "cores": threads, "kind": "port",
            "sample": "%d of %d instances x %d sweeps, OpenMP over instances, %d threads, %.1f s"
                      % (nb, stage.shape[0], reps, threads, t),
            "ok": bool((bo.status == 1).all())}, bo


def _single_instance_cpu_rows(budget_s=4.0):
    """BASELINE.md section 4: single-instance CPU rows -- C1 dims (nx6 nu3 N100) and the reference bench's
    native shape (nx36 nu12 nc32, bench/gar-riccati.cpp:19-22) serial and leg-split with 2/4/6 threads
    (bench/gar-riccati.cpp:87-90), timed on the oracle's restatement of both solvers."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import gen
    from oracle import gar_oracle as orc
    rows = []
    cases = [("c1 nx6 nu3 N100", 6, 3, 0, 100, 1e-11, "conditioned")]
    for N in (16, 64, 256, 1024):
        cases.append(("native nx36 nu12 nc32 N%d" % N, 36, 12, 32, N, 1e-11, "reference"))
    per = budget_s / (len(cases) * 4)
    for name, nx, nu, nc, N, mu, style in cases:
        rng = np.random.default_rng(7)
        prob = gen.generate_lq_problem(rng, rng.standard_normal(nx), N, nx, nu, 0, nc, singular=(style == "reference"),
                                       conditioned=(style != "reference"), control_rows=False)
        for threads in (1, 2, 4, 6):
            op = orc.OracleProblem(prob.copy())
            if threads == 1:
                sv = orc.ProximalRiccatiSolver(op)
            else:
                if N + 1 < threads:
                    continue
                sv = orc.ParallelRiccatiSolver(op, threads, threaded=True)
            sol = orc.OracleSolution(op)
            sv.backward(mu)
            sv.forward(sol)  # warm-up
            reps, t0 = 0, time.perf_counter()
            while True:
                sv.backward(mu)
                sv.forward(sol)
                reps += 1
                dt = time.perf_counter() - t0
                if dt >= per or reps >= 2000:
                    break
            rows.append({"case": name, "threads": threads, "ms_per_sweep": 1e3 * dt / reps,
                         "knots_per_s": (N + 1) * reps / dt})
    return rows


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (oracle port; the reference
    cannot be compiled in this image) on the box's host cores, same workload/metric.
    One step = one sweep over a bounded sample of the workload (up to 1024 of its instances, fewer when an
    instance is expensive: the whole run stays near half a minute); the thread count is the faster of "every
    hardware thread" and "half of them".  The timed window is exactly --steps sweeps.  With --ref-seconds S
    (the product arm's cpu_baseline) it is sized by time instead: the figure is the MEDIAN of 5 timed repeats,
    each of max(0.7 s, S / 5) worth of sweeps, so a single slow repeat (thread start-up, a noisy neighbour)
    does not move it."""
    if rank != 0:
        return
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    from oracle import gar_oracle as orc
    # every host core (torchrun exports OMP_NUM_THREADS=1 to its workers: ask explicitly)
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    allthr = max(orc.num_threads(), avail)
    # Bounded sample: a probe of one instance per thread gives the time of one "round"; the sample is as many
    # rounds as keep 5 x --steps sweeps near 25 s (C2: the cap of 1024 instances; C5: one or two rounds).
    def make(nb_):
        a = [x.numpy() for x in synth_batch_torch(torch, nb_, HORIZON, NX, NU, "cpu", 1234, NC)]
        return orc.BatchedOracle(NX, NU, NC, NCT, NX, HORIZON, nb_, *a)
    probe = make(min(allthr, BATCH))
    probe.sweep(MUEQ, reps=1, nthreads=allthr)
    t_round = min(probe.sweep(MUEQ, reps=1, nthreads=allthr) for _ in range(2))
    rounds = max(1, int(25.0 / (5.0 * max(args.steps, 1) * max(t_round, 1e-5))))
    nb = max(min(allthr, BATCH), min(1024, BATCH, rounds * allthr))
    bo = make(nb)
    # thread count: all visible hardware threads or half of them (one per physical core) -- whichever is
    # faster on this box is the CPU's best figure (measured: 64 threads beat 128 by 1.6x on a 2 x 32-core host)
    cand = [allthr] + ([allthr // 2] if allthr >= 16 else [])
    best = {}
    for th in cand:
        bo.sweep(MUEQ, reps=1, nthreads=th)
        best[th] = min(bo.sweep(MUEQ, reps=1, nthreads=th) for _ in range(3))
    threads = min(best, key=best.get)
    # warm-up: W sweeps and at least 1.5 s (the worker threads' first sweeps run far below the
    # sustained pace: thread start-up, allocator arenas, first touch)
    t1, tw, nw = 1e9, 0.0, 0
    while nw < max(args.warmup, 1) or tw < 1.5:
        dt = bo.sweep(MUEQ, reps=1, nthreads=threads)
        t1, tw, nw = min(t1, dt), tw + dt, nw + 1
    if args.ref_seconds > 0:
        repeats = 5
        steps = int(max(0.7, args.ref_seconds / 5.0) / max(t1, 1e-5)) + 1
    else:
        repeats, steps = 1, args.steps
    rates, total_t = [], 0.0
    for _ in range(repeats):
        t = bo.sweep(MUEQ, reps=steps, nthreads=threads)
        total_t += t
        rates.append(nb * (HORIZON + 1) * steps / t)
    rates.sort()
    v = rates[repeats // 2]
    assert bool((bo.status == 1).all())
    cpu = {"value": v, "unit": "knots/s", "cores": threads, "kind": "port",
           "min": rates[0], "max": rates[-1], "repeats": repeats,
           "sample": "%d of %d instances per step, %d repeat(s) x %d steps (%.1f s in all), OpenMP over instances on %d "
                     "threads (%d hardware threads visible; thread counts tried: %s), median of the repeats"
                     % (nb, BATCH, repeats, steps, total_t, threads, avail,
                        ", ".join("%d: %.1f ms/sweep" % (k, 1e3 * v_) for k, v_ in best.items()))}
    if args.cpu_extra:
        try:
            cpu["single_instance"] = _single_instance_cpu_rows()
        except Exception as e:  # the extra rows never break the arm
            cpu["single_instance"] = "failed: %r" % (e,)
    line = {"metric": "riccati_knots_per_sec", "value": v, "unit": "knots/s", "n_gpus": args.gpus,
            "steps": steps * repeats, "warmup": nw, "ms_per_step": 1e3 * total_t / (repeats * steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "step_sample": "%d instances per step" % nb,
                       "mueq": MUEQ, "note": "reference cannot be built here (no Eigen); "
                       "restated C++ port of gar::ProximalRiccatiSolver, OpenMP over instances"},
            "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": "knots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def parity_sample(gar, solver, stage, term, G0, g0, nsamp=16):
    """Correctness gate printed with every timing (BASELINE.md section 4): max over (instance, t) of the
    relative Frobenius error of K_t, k_t, Vxx_t of `nsamp` instances spread over the batch against the CPU
    oracle on the same inputs.  Outside the timed region."""
    import numpy as np
    from oracle import gar_oracle as orc
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import gen
    B, N = stage.shape[0], HORIZON
    idx = sorted(set(int(round(i * (B - 1) / max(nsamp - 1, 1))) for i in range(nsamp)))
    h = [a[idx].cpu().numpy() for a in (stage, term, G0, g0)]
    bo = orc.BatchedOracle(NX, NU, NC, NCT, NX, N, len(idx), *h)
    bo.sweep(MUEQ)
    ref = bo.get()
    worst = {"K": 0.0, "k": 0.0, "Vxx": 0.0}
    nr = NU + NC + NX
    for j, b in enumerate(idx):
        fb = np.empty(N * nr * NX)
        ff = np.empty(N * nr)
        V = np.empty((N + 1) * NX * NX)
        solver.get_range_into(gar.OUT_FB, b, 1, 0, N, fb, gar.AB2_HOST)
        solver.get_range_into(gar.OUT_FF, b, 1, 0, N, ff, gar.AB2_HOST)
        solver.get_range_into(gar.OUT_VXX, b, 1, 0, N + 1, V, gar.AB2_HOST)
        solver.synchronize()
        fb, ff = fb.reshape(N, nr, NX), ff.reshape(N, nr)
        V = V.reshape(N + 1, NX, NX).transpose(0, 2, 1)
        for t in range(N):
            worst["K"] = max(worst["K"], gen.rel_fro(fb[t, :NU], ref["fb"][j, t, :NU]))
            worst["k"] = max(worst["k"], gen.rel_fro(ff[t, :NU], ref["ff"][j, t, :NU]))
        for t in range(N + 1):
            worst["Vxx"] = max(worst["Vxx"], gen.rel_fro(V[t], ref["Vxx"][j, t]))
    tolk = max(1e-10, 2.4e-16 / MUEQ) if NC > 0 else 1e-10
    worst.update({"instances": len(idx), "tolerance": 1e-10, "tolerance_K_constrained": tolk,
                  "ok": bool(worst["Vxx"] <= 1e-10 and worst["K"] <= tolk and worst["k"] <= tolk),
                  "against": "oracle/gar_oracle (CPU restatement of the reference; parity unpinned)"})
    return worst


DUMP_BYTES = 60 * 10 ** 6  # the sample's data; with the .npy headers it stays below 64 MB
DUMP_SEED = 2024


def dump_outputs(gar, solver, outdir):
    """Writes what the last sweep returned to its caller -- gains ff, fb, value function Vxx, vx, terminal
    gains ffT, fbT and the primal-dual trajectory xs, us, vs, vsT, lbd0, lbdas -- as <outdir>/<name>.npy
    (float64, Vxx indexed [b, t, i, j]), so that two builds can be compared output for output.  A full batch
    is too large to keep: every array holds the same instances, a seeded sample of the batch (sorted, the
    same for every build at a given batch size) as large as fits DUMP_BYTES in all; idx.npy holds their
    batch indices (as float64)."""
    import numpy as np
    outs = {"ff": gar.OUT_FF, "fb": gar.OUT_FB, "Vxx": gar.OUT_VXX, "vx": gar.OUT_VX, "ffT": gar.OUT_FFT,
            "fbT": gar.OUT_FBT, "xs": gar.OUT_XS, "us": gar.OUT_US, "vs": gar.OUT_VS, "vsT": gar.OUT_VST,
            "lbd0": gar.OUT_LBD0, "lbdas": gar.OUT_LBDAS}
    shapes = {k: solver.out_shape(w) for k, w in outs.items() if int(np.prod(solver.out_shape(w))) > 0}
    B = solver.dims.batch
    per_instance = sum(int(np.prod(s[1:])) for s in shapes.values()) * 8
    n = max(1, min(B, DUMP_BYTES // per_instance))
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(B, n, replace=False))
    per_instance_outs = (gar.OUT_FFT, gar.OUT_FBT, gar.OUT_VST, gar.OUT_LBD0)
    os.makedirs(outdir, exist_ok=True)
    np.save(os.path.join(outdir, "idx.npy"), idx.astype(np.float64))
    for name, shape in shapes.items():
        knots = 1 if outs[name] in per_instance_outs else shape[1]
        a = np.empty((n,) + tuple(shape[1:]))
        for j, b in enumerate(idx):
            solver.get_range_into(outs[name], int(b), 1, 0, knots, a[j], gar.AB2_HOST)
        solver.synchronize()
        if outs[name] == gar.OUT_VXX:  # column-major blocks in memory
            a = a.transpose(0, 1, 3, 2)
        np.save(os.path.join(outdir, name + ".npy"), np.ascontiguousarray(a))


def bind_to_gpu_numa(local):
    """Pin this process to the CPUs closest to its GPU (NVML's ideal-CPU mask = the GPU's NUMA node)
    BEFORE any pinned host memory is allocated, so the e2e staging buffers land on that node (first
    touch) and the 8 ranks do not all pull through one socket's PCIe root."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1 and 64 * w + b < ncpu]
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"bound": True, "cpus": len(cpus), "first": cpus[0], "last": cpus[-1]}
        return {"bound": False, "why": "empty affinity mask"}
    except Exception as e:
        return {"bound": False, "why": repr(e)[:80]}


def main():
    global NX, NU, NC, NCT, HORIZON, BATCH, MUEQ, WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--variant", type=int, default=-1)
    ap.add_argument("--e2e-chunks", type=int, default=0, help="slices of the pipelined e2e call (0 = auto)")
    ap.add_argument("--stagger-ns", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--ref-seconds", type=float, default=0.0)
    ap.add_argument("--cpu-extra", action="store_true", help="single-instance CPU rows (BASELINE.md section 4)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--strong", default="c4", help="also time this config's FULL batch split over the ranks (none = skip)")
    ap.add_argument("--strong-legs", type=int, default=0, help="parallel-in-time legs for the strong-scaling run")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="the one exchange: fused pack + NVLink peer-memory all-gather, or pack kernel + ncclAllGather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the product arm's outputs; --impl reference has none to write")
    if args.config != "c2":
        NX, NU, NC, NCT, HORIZON, BATCH, MUEQ, WORKLOAD = CONFIGS[args.config]
        if args.batch == 4096:
            args.batch = BATCH
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    numa = bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    import aligator_b200.gar as gar

    B, N = args.batch, HORIZON
    stage, term, G0, g0 = synth_batch_torch(torch, B, N, NX, NU, dev, 1234 + rank, NC)
    solver = gar.CudaRiccatiBatch(NX, NU, NC, NCT, NX, N, B, device=local, variant=args.variant,
                                  stagger_ns=args.stagger_ns, ctas_per_sm=args.ctas_per_sm)
    stream = torch.cuda.current_stream().cuda_stream
    solver.set_problem(stage, term, G0, g0, memspace=gar.AB2_DEVICE, stream=stream)
    # first-step policy [K0 | k0] per instance: the one all-gather when the batch shards.
    # The gather of sweep i runs on a side stream and overlaps sweep i+1 (two buffers).
    pol = [torch.empty(B, NU, NX + 1, dtype=torch.float64, device=dev) for _ in range(2)]
    pol_all = [torch.empty(world * B, NU, NX + 1, dtype=torch.float64, device=dev) for _ in range(2)] \
        if world > 1 else None
    main = torch.cuda.current_stream()
    side = torch.cuda.Stream() if world > 1 else None
    gathered = [None, None]
    step_no = [0]

    from aligator_b200 import sharding
    peer = world > 1 and args.gather == "peer"
    peer_note = None
    if peer:
        try:  # (collective-safe: every rank raises or none does)
            solver.peer_gather_setup(dist, rank, world)
        except gar.GarError as e:  # no CUDA IPC / peer access on this box: the library collective takes over
            peer, peer_note = False, str(e)
    waited = [None]

    def step():
        solver.sweep(MUEQ, stream=stream)
        if peer:
            # the one exchange, fused: the pack kernel stores [K0 | k0] straight into every rank's
            # receive buffer over NVLink (no NCCL kernel); arrival is awaited on the side stream,
            # overlapping the next sweep; the next pack waits for that (its ack says "consumed")
            if len(waited) >= 3 and waited[-2] is not None:
                main.wait_event(waited[-2])  # the arrival (and consumption) of the gather TWO steps back
            solver.policy_allgather(stream=stream)
            side.wait_stream(main)
            solver.policy_allgather_wait(stream=side.cuda_stream)
            ev = torch.cuda.Event()
            ev.record(side)
            waited.append(ev)
            del waited[:-3]
        elif world > 1:  # the one exchange: all-gather of the first-step policy [K0 | k0]
            i = step_no[0] & 1
            step_no[0] += 1
            if gathered[i] is not None:
                main.wait_event(gathered[i])  # the gather that last read pol[i] is done
            solver.first_step_policy_into(pol[i], stream=stream)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                sharding.all_gather_policy(torch, dist, pol[i], world, out=pol_all[i])
                ev = torch.cuda.Event()
                ev.record(side)
            gathered[i] = ev

    def join():  # every gather issued so far has completed before the timer stops
        if side is not None:
            main.wait_stream(side)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    assert int(solver.status().max()) == 0, "factorisation failure flagged"
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = solver.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    join()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = solver.launch_count() - l0
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    knots = B * (N + 1) * world
    value = knots / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(gar, solver, args.dump_outputs)

    # ---- e2e through the C ABI with host (pinned) buffers ----
    e2e = None
    if not args.no_e2e:
        hs = [torch.empty(a.shape, dtype=torch.float64, pin_memory=True) for a in (stage, term, G0, g0)]
        for h, a in zip(hs, (stage, term, G0, g0)):
            h.copy_(a)
        outs = (gar.OUT_XS, gar.OUT_US, gar.OUT_LBDAS, gar.OUT_LBD0, gar.OUT_FF, gar.OUT_FB)
        hout = [torch.empty(max(int(np.prod(solver.out_shape(w))), 1), dtype=torch.float64,
                            pin_memory=True) for w in outs]
        s2 = gar.CudaRiccatiBatch(NX, NU, NC, NCT, NX, N, B, device=local, variant=args.variant,
                                  stagger_ns=args.stagger_ns, ctas_per_sm=args.ctas_per_sm)

        # Q and R of every knot cross PCIe as lower triangles (ab2_gar_sweep_host_sym): the path is PCIe-bound, so
        # the 16 % fewer bytes are 16 % less time.  The full-record call is timed beside it.
        nsym = int(gar.lib().ab2_gar_stage_record_doubles_sym(NX, NU, NC))
        hsym = torch.empty(B * N * nsym, dtype=torch.float64, pin_memory=True)
        s2.pack_stage_sym(hs[0].numpy(), out=hsym.numpy())

        def run_e2e(sym):
            def e2e_step():
                # one call of the public host-buffer API: upload, sweep and download pipelined
                # over slices of the batch (PCIe full duplex: max(H2D, D2H) instead of the sum)
                if sym:
                    s2.sweep_host_sym(hsym, hs[1], hs[2], hs[3], MUEQ, dict(zip(outs, hout)),
                                      nchunks=args.e2e_chunks, stream=stream)
                else:
                    s2.sweep_host(hs[0], hs[1], hs[2], hs[3], MUEQ, dict(zip(outs, hout)),
                                  nchunks=args.e2e_chunks, stream=stream)
                s2.synchronize(stream)

            e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2e_step()
            barrier()
            dt = (time.perf_counter() - t0) / args.e2e_steps
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        dt_full = run_e2e(False)
        dt = run_e2e(True)
        # the host-buffer path returns what the device-resident arm computed (same inputs): checked outside the timing
        xs_dev = solver.get(gar.OUT_XS)
        xs_e2e = hout[0].numpy()[:xs_dev.size].reshape(xs_dev.shape)
        e2e_err = float(np.abs(xs_e2e - xs_dev).max() / max(np.abs(xs_dev).max(), 1e-300))
        h2d_full = sum(h.numel() for h in hs) * 8
        h2d = h2d_full - hs[0].numel() * 8 + hsym.numel() * 8
        d2h = sum(int(np.prod(solver.out_shape(w))) for w in outs) * 8
        arms = {"ab2_gar_sweep_host_sym: Q, R uploaded as lower triangles; upload/sweep/download pipelined over batch slices":
                (dt, h2d),
                "ab2_gar_sweep_host: upload/sweep/download pipelined over batch slices": (dt_full, h2d_full)}
        api = min(arms, key=lambda k: arms[k][0])  # the headline is the faster public call; the other is listed beside it
        other = [k for k in arms if k != api][0]
        e2e = {"value": knots / arms[api][0], "unit": "knots/s", "h2d_bytes_per_step": arms[api][1],
               "d2h_bytes_per_step": d2h, "ms_per_step": arms[api][0] * 1e3, "steps": args.e2e_steps,
               "reads": "xs,us,lbdas,lbd0,ff,fb (what solver-proxddp.hxx:610-632 consumes)",
               "api": api, "xs_vs_device_arm": e2e_err,
               "other_api": {"api": other, "value": knots / arms[other][0], "ms_per_step": arms[other][0] * 1e3,
                             "h2d_bytes_per_step": arms[other][1]}}
        s2.close()

    # ---- e2e_device: the device-resident inner loop (INTEGRATION.md section 3b): the knots are ASSEMBLED on the
    # device from resident derivative buffers (updateLQSubproblem), swept, and the line-search consumers
    # (directional derivative, linear step) run there too; only [batch] scalars cross PCIe per iteration ----
    e2e_device = None
    if not args.no_e2e and NC == 0:
        o = 0
        fld = {}
        for name, n in (("Jx", NX * NX), ("Ju", NX * NU), ("slack", NX), ("Lxx", NX * NX), ("Lxu", NX * NU),
                        ("Luu", NU * NU), ("Lx", NX), ("Lu", NU)):
            fld[name] = stage[:, :, o:o + n].contiguous()
            o += n
        fld.update(Lxx_N=term[:, :NX * NX].contiguous(), Lx_N=term[:, NX * NX:NX * NX + NX].contiguous(), G0=G0, g0=g0)
        s4 = gar.CudaRiccatiBatch(NX, NU, NC, NCT, NX, N, B, device=local, variant=args.variant)
        Lxs = torch.randn(B, N + 1, NX, dtype=torch.float64, device=dev)
        Lus = torch.randn(B, N, NU, dtype=torch.float64, device=dev)
        cur = {k: torch.zeros(solver.out_shape(w), dtype=torch.float64, device=dev)
               for k, w in dict(xs=gar.OUT_XS, us=gar.OUT_US, vs=gar.OUT_VS, vsT=gar.OUT_VST, lam0=gar.OUT_LBD0,
                                lams=gar.OUT_LBDAS).items()}
        trial = {k: torch.empty_like(v) for k, v in cur.items()}

        def dev_step():
            s4.assemble(fld, 0.0, 1.0, stream=stream)
            s4.sweep(MUEQ, stream=stream)
            s4.linear_step(1.0, cur, trial, stream=stream)
            return s4.directional_derivative(Lxs, Lus, stream=stream)  # [batch] doubles to the host, synchronises

        dev_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            d1 = dev_step()
        barrier()
        dtd = (time.perf_counter() - t0) / args.e2e_steps
        td = torch.tensor([dtd], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        dtd = float(td.item())
        e2e_device = {"value": knots / dtd, "unit": "knots/s", "ms_per_step": dtd * 1e3, "h2d_bytes_per_step": 0,
                      "d2h_bytes_per_step": B * 8, "steps": args.e2e_steps,
                      "pipeline": "ab2_gar_assemble (updateLQSubproblem on device) -> ab2_gar_sweep -> ab2_gar_linear_step "
                                  "-> ab2_gar_directional_derivative; only the [batch] directional derivatives return",
                      "finite": bool(np.isfinite(d1).all())}
        s4.close()

    # ---- strong scaling: the FULL batch of BASELINE config 4 (nx14 nu7 N200, 2048 instances) split over
    # the ranks (SURVEY 8e: 2048 -> 1024/512/256 per GPU), same fused exchange; every rank measures ----
    strong = None
    if args.strong in CONFIGS:
        snx, snu, snc, snct, sN, sB, smu, swl = CONFIGS[args.strong]
        b0, b1 = sharding.shard_range(sB, rank, world)
        sb = b1 - b0
        sst = synth_batch_torch(torch, sb, sN, snx, snu, dev, 4321 + rank, snc)
        s3 = gar.CudaRiccatiBatch(snx, snu, snc, snct, snx, sN, sb, device=local, legs=args.strong_legs)
        s3.set_problem(*sst, memspace=gar.AB2_DEVICE, stream=stream)
        speer = peer and sb * world == sB
        if speer:
            s3.peer_gather_setup(dist, rank, world)
        sw = [None]

        def sstep():
            s3.sweep(smu, stream=stream)
            if speer:
                if len(sw) >= 3 and sw[-2] is not None:
                    main.wait_event(sw[-2])
                s3.policy_allgather(stream=stream)
                side.wait_stream(main)
                s3.policy_allgather_wait(stream=side.cuda_stream)
                ev = torch.cuda.Event()
                ev.record(side)
                sw.append(ev)
                del sw[:-3]

        for _ in range(max(args.warmup, 3)):
            sstep()
        join()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            sstep()
        join()
        f1.record()
        barrier()
        t3 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        sms = float(t3.item()) / args.steps
        ok3 = int(s3.status().max()) == 0
        strong = {"workload": swl + " -- TOTAL batch %d split over %d GPU(s)" % (sB, world), "scaling": "strong",
                  "batch_per_gpu": sb, "legs": args.strong_legs, "ms_per_step": sms,
                  "value": sB * (sN + 1) / (sms * 1e-3), "unit": "knots/s", "ok": ok3,
                  "exchange": "fused pack + NVLink peer all-gather of [K0|k0]" if speer else ("none" if world == 1 else "nccl/none"),
                  "kernel": s3.kernel_info()}
        s3.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    parity = None
    if not args.no_parity:
        try:
            parity = parity_sample(gar, solver, stage, term, G0, g0)
        except Exception as e:
            parity = {"ok": False, "error": repr(e)}

    # ---- roofline of the (single) kernel ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    bpk = bytes_per_knot(NX, NU, NC)
    kernel_ms = ms_per_step  # one launch per step; the all-gather (N>1) is outside this figure at N=1
    achieved = B * (N + 1) * bpk / (kernel_ms * 1e-3) / 1e9
    traffic = None  # ncu dram bytes per launch of THIS config's kernel (profiles/traffic.json), else null
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            ent = json.load(open(tp)).get(args.config)
            if ent and ent.get("batch") == B:
                traffic = ent.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_knot": bpk, "kernel": "riccati_sweep_kernel",
                "kernel_ms": kernel_ms}
    if args.config == "c5":
        # ~11 flop/B: the bound of this shape is the FP64 pipe, not HBM.  Peak = the DFMA / DMMA rate measured on
        # this GPU with tools/micro/fp64_rates under ncu (profiles/r02_fp64_rates_ncu.csv: 0.24 DMMA m8n8k4 per
        # clock per SM = 61.4 FMA/clk/SM, tensor pipe 99.8 % active) x 148 SMs x 1.965 GHz = 35.7 TFLOP/s.
        fpk = 4 * NX ** 3 + 8 * NX * NX * NU + 4 * NX * NU * NU + NU ** 3 / 3.0 + 2 * NU * NU * (NX + 1) \
            + 2 * (NU + NX) * NX + 2 * NX * NX   # SURVEY 8(d) flops per knot (backward + forward)
        tf = B * (N + 1) * fpk / (kernel_ms * 1e-3) / 1e12
        roofline = {"bound": "fp64", "achieved": tf, "peak": 35.7, "unit": "TFLOP/s", "frac": tf / 35.7,
                    "traffic": traffic, "peak_source": "measured DFMA = DMMA rate (tools/micro/fp64_rates, profiles/r02_fp64_rates_ncu.csv)",
                    "algorithmic_flops_per_knot": fpk, "kernel": "riccati_block_kernel (CTA per instance)",
                    "kernel_ms": kernel_ms, "hbm": {"achieved": achieved, "peak": peak, "frac": achieved / peak}}

    cpu = None
    if not args.no_cpu:
        # The CPU arm runs in a fresh process: inside this one torch's own OpenMP runtime
        # competes with the oracle's thread pool (measured 5x slower), which would flatter
        # the GPU.  Same code path as `--impl reference`, sized to ~12 s of CPU work.
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference",
                            "--config", args.config, "--warmup", "2", "--ref-seconds", "12", "--cpu-extra"],
                           capture_output=True, text=True)
        try:
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception:
            cpu = {"value": None, "unit": "knots/s", "cores": None, "kind": "port",
                   "sample": "reference arm failed: " + (r.stderr or r.stdout)[-200:]}

    line = {"metric": "riccati_knots_per_sec", "value": value, "unit": "knots/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "nx": NX, "nu": NU, "nc": NC, "horizon": N,
                       "batch_per_gpu": B, "mueq": MUEQ, "parallelism": "batch-sharded x%d" % world,
                       "generator": "SURVEY 8(d) conditioned variant, counter-seeded per rank",
                       "l2": "inputs+outputs per sweep (%.2f GB) exceed the 126 MB L2; no flush needed"
                             % ((stage.numel() * 8 + B * (N + 1) * 8 * ((NU + NC + NX) * (NX + 1) + NX * NX + NX)) / 1e9),
                       "kernel": solver.kernel_info(), "variant": args.variant, "numa": numa,
                       "exchange": ("fused pack + NVLink peer-memory all-gather of [K0|k0] (no NCCL on the data path)"
                                    if peer else (("ncclAllGather of [K0|k0]" + (" (peer memory unavailable: %s)" % peer_note if peer_note else ""))
                                                  if world > 1 else "none (1 GPU)"))},
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clk, "e2e": e2e,
            "gpu_launches": launches, "parity": parity, "strong": strong, "e2e_device": e2e_device}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
