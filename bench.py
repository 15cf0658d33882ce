#!/usr/bin/env python
"""bench.py -- candidate (whole+safe pair) trajectory solves per second on BASELINE.json's configurations.

Default workload = BASELINE config 4 as written: random-forest corridors (JPS3D + convex decomposition on the host,
committed as bench_data/cfg4_forest.npz by tools/make_cfg4_fixture.py), PAIRED whole + safe solve: per corridor the
whole sweep (N=10, 3 polytopes, 16 time allocations x 64 assignments = 1024 candidates, final position pinned), the
genNewTraj selection, R = sample (int)(0.6 n) of the winner, then the safe sweep FROM R (N=10, 4 polytopes, 1024
candidates, final position free) -- two dependent launches per batch, chained on the device (fq_replan_pairs_dev).
One pass = 64 corridors = 65 536 pairs per GPU; one step = --inner passes over a ring of distinct batches.

value : pairs/s, inputs resident in HBM, CUDA-event timed, max over ranks.  N > 1: every rank runs its own 64 corridors
        per pass (weak scaling) and every chain ends with the path's one collective, an NCCL all-gather of the
        per-corridor result records inside the library; "strong" reports the same 65 536 pairs split over the ranks.
e2e   : the same through the host-pointer C ABI (fq_replan_pairs_async on two contexts) from pinned host arrays.
other_configs : BASELINE configs 2, 3 and 5 as written (single-kind batches), each with kernel time, roofline, parity.
--impl reference : the CPU arm (Gurobi itself is unavailable): the CPU port of the same chain on all host threads.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SEG = 10
BYTES_PER_CAND = {10: 8 * (9 + 9 + 3 + 1) + 10 + 1 + 8, 15: 8 * (9 + 9 + 3 + 1) + 15 + 1 + 8}   # SURVEY 8(d): 195 / 200 B
METRIC = "candidate (whole+safe pair) trajectory solves/sec"
CFG4_NAME = ("cfg4: random-forest corridors (host JPS3D + convex decomposition), paired whole (N=10, P=3) + safe (N=10, P=4, "
             "x0 = whole winner's sample at 60 % of the horizon) solve, 64 corridors x 1024 pairs = 65 536 pairs per pass")
FIXTURE = os.path.join(ROOT, "bench_data", "cfg4_forest.npz")
PAIR_KEYS = ["x0", "xf_whole", "xf_safe", "lim", "poly_ofs_whole", "face_ofs_whole", "Ab_whole", "poly_ofs_safe",
             "face_ofs_safe", "Ab_safe", "factors_whole", "sigmas_whole", "factors_safe", "sigmas_safe"]


# ----------------------------------------------------------------------------------------------------------------------
# workloads (numpy only: both arms use these)
# ----------------------------------------------------------------------------------------------------------------------
_fx = None


def load_cfg4(start, count):
    """Corridors [start, start+count) (cyclic) of the committed config-4 fixture as a pair-workload dict (the layout of
    fq_pair_args; see faster_b200.capi.make_pair_workload)."""
    global _fx
    if _fx is None:
        _fx = dict(np.load(FIXTURE))
    f = _fx
    n_all = int(f["meta"][0])
    idx = [(start + i) % n_all for i in range(count)]

    def sub(po, fo, Ab):
        npo, nfo, rows = [0], [0], []
        for j in idx:
            for p in range(po[j], po[j + 1]):
                rows.append(Ab[fo[p]:fo[p + 1]])
                nfo.append(nfo[-1] + fo[p + 1] - fo[p])
            npo.append(npo[-1] + po[j + 1] - po[j])
        nfo = np.asarray(nfo, np.int32); npo = np.asarray(npo, np.int32)
        mf = int(max(nfo[npo[j + 1]] - nfo[npo[j]] for j in range(count)))
        return npo, nfo, np.ascontiguousarray(np.vstack(rows)), mf, int(np.diff(nfo).max())
    pw, fw, Aw, mfw, mpfw = sub(f["poly_ofs_whole"], f["face_ofs_whole"], f["Ab_whole"])
    ps, fs, As, mfs, mpfs = sub(f["poly_ofs_safe"], f["face_ofs_safe"], f["Ab_safe"])
    return dict(n_prob=count, N_whole=int(f["meta"][1]), N_safe=int(f["meta"][2]), DC=float(f["DC"]), r_fraction=float(f["r_fraction"]),
                x0=np.ascontiguousarray(f["x0"][idx]), xf_whole=np.ascontiguousarray(f["xf_whole"][idx]),
                xf_safe=np.ascontiguousarray(f["xf_safe"][idx]), lim=np.ascontiguousarray(f["lim"][idx]),
                poly_ofs_whole=pw, face_ofs_whole=fw, Ab_whole=Aw, poly_ofs_safe=ps, face_ofs_safe=fs, Ab_safe=As,
                factors_whole=f["factors_whole"].copy(), sigmas_whole=f["sigmas_whole"].copy(),
                factors_safe=f["factors_safe"].copy(), sigmas_safe=f["sigmas_safe"].copy(),
                max_faces_whole=mfw, max_poly_faces_whole=mpfw, max_faces_safe=mfs, max_poly_faces_safe=mpfs,
                R_oracle=np.ascontiguousarray(f["R_oracle"][idx]))


def pairs_per_pass(w):
    return w["n_prob"] * len(w["factors_whole"]) * len(w["sigmas_whole"])


SINGLE = {   # BASELINE configs 2, 3, 5 as SURVEY 8(d) specifies them
    "cfg2": dict(name="cfg2: whole-trajectory QP, N=10, 3 polytopes, 1024 candidates per corridor (16 dt x 64 sigma)",
                 N=10, P=3, ff=True, profile="uav", n_dt=16, n_sig=64, corridors=64, seed=2000),
    "cfg3": dict(name="cfg3: safe-trajectory MIQP candidates, N=10, 4 polytopes, 8192 per corridor (32 dt x 256 sigma)",
                 N=10, P=4, ff=False, profile="uav", n_dt=32, n_sig=256, corridors=8, seed=3000),
    "cfg5": dict(name="cfg5: ground robot (v 1.4, a 1.4, j 5.0), N=15, 8 narrow polytopes, 32 768 per corridor (16 dt x 2048 sampled sigma)",
                 N=15, P=8, ff=True, profile="ground", n_dt=16, n_sig=2048, corridors=2, seed=5000),
}


def make_single(cfg, n_corr, dt_initial):
    """Synthetic corridors of a single-kind configuration laid out for fq_solve_multi.  dt_initial(x0, xf, lim, N) is the
    arm's own getDTInitial (product library or oracle), so that neither arm needs the other's code."""
    from faster_b200 import corridor as cr           # pure numpy module
    N, P = cfg["N"], cfg["P"]
    if cfg["n_sig"] >= 1024:
        sig = cr.sample_monotone_sigmas(N, P, cfg["n_sig"], np.random.default_rng(cfg["seed"]))
    else:
        allm = cr.monotone_sigmas(N, P)
        sig = allm[np.linspace(0, len(allm) - 1, cfg["n_sig"]).round().astype(int)]
    cand = cfg["n_dt"] * cfg["n_sig"]
    x0 = np.zeros((n_corr, 9)); xf = np.zeros((n_corr, 9)); lim = np.zeros((n_corr, 3))
    po, fo, rows = [0], [0], []
    dts = np.zeros((n_corr, cand)); sigs = np.zeros((n_corr, cand, N), np.uint8)
    for c in range(n_corr):
        pb = cr.make_corridor(cfg["seed"] + c, P, N, cfg["profile"], cfg["ff"])
        x0[c], xf[c], lim[c] = pb["x0"], pb["xf"], pb["lim"]
        for A, b in pb["polys"]:
            rows.append(np.hstack([A, b[:, None]])); fo.append(fo[-1] + len(b))
        po.append(po[-1] + P)
        base = max(dt_initial(pb["x0"], pb["xf"], pb["lim"], N), 2 * pb["DC"])
        dts[c] = np.repeat(np.arange(1.0, cfg["n_dt"] + 1) * base, cfg["n_sig"])        # factors 1..n_dt (faster.cpp:57)
        sigs[c] = np.tile(sig, (cfg["n_dt"], 1))
    fo = np.asarray(fo, np.int32); po = np.asarray(po, np.int32)
    return dict(N=N, ff=cfg["ff"], n_prob=n_corr, cand=cand, x0=x0, xf=xf, lim=lim, poly_ofs=po, face_ofs=fo,
                Ab=np.ascontiguousarray(np.vstack(rows)), cand_ofs=(np.arange(n_corr + 1) * cand).astype(np.int32),
                dt=dts.reshape(-1), sigma=sigs.reshape(-1, N),
                max_faces=int(max(fo[po[j + 1]] - fo[po[j]] for j in range(n_corr))), max_poly_faces=int(np.diff(fo).max()))


N_DT, N_SIG, CAND = 16, 64, 1024
STRONG_CONTEXTS = 6      # chains in flight per GPU for the strong-scaling leg (small shards)


def make_workload(n_corr, seed0, kind):
    """Round 1's synthetic "cfg2-pairs" batches (whole: P=3, final position pinned; safe: P=4, free), still used by the
    stress and modelling tools under tools/: make_single's layout plus the corridor dicts."""
    from faster_b200 import capi, corridor as cr
    cfg = dict(SINGLE["cfg2"], seed=seed0) if kind == "whole" else dict(SINGLE["cfg2"], P=4, ff=False, seed=seed0)
    w = make_single(cfg, n_corr, capi.dt_initial)
    w["kind"] = kind
    w["probs"] = [cr.make_corridor(seed0 + c, cfg["P"], cfg["N"], cfg["profile"], cfg["ff"]) for c in range(n_corr)]
    return w


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append((float(f[0]), float(f[1]), f[2:]))
            except Exception:
                pass
            time.sleep(0.01)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i, v in enumerate(s[2]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median([s[0] for s in self.samples])), "sm_max_mhz": self.samples[0][1],
                "reasons": reasons, "samples": len(self.samples)}


def cfg4_config(world, C):
    """Identical for both arms (the driver compares the two lines' configs)."""
    return {"workload": CFG4_NAME, "corridors_per_gpu_per_pass": C, "pairs_per_pass_per_gpu": C * 1024,
            "l2": "flushed between timed steps (256 MiB memset outside the per-step events); a step cycles through a ring of distinct batches",
            "parallelism": ("corridor shards per rank + one NCCL all-gather of the per-corridor result records (inside the library)"
                            if world > 1 else "single GPU")}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm
# ----------------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm may really use: the scheduler affinity and the cgroup CPU quota of this container, not the
    machine's core count (a 1-GPU slice of an 8-GPU host gets a slice of its cores)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


CPU_NOTE = ("tuned CPU port of the GPU kernel's algorithm (oracle/fq_cpu_port.c: plan tables, normalised pivoting, thin "
            "factorisation, persistent thread pool with dynamic claiming, AVX2) driving the same chain; Gurobi itself is unavailable")


def cpu_pair_rate(n_corr, threads, min_seconds, start=256, fast=True):
    """The CPU arm on a bounded sample of the same fixture.  -> (pairs/s, sample text)."""
    from oracle import pair_oracle, pyoracle as po
    ws = [load_cfg4(start + n_corr * k, n_corr) for k in range(4)]
    run = (lambda w: po.replan_pairs_port(w, threads)) if fast else (lambda w: pair_oracle.replan_pairs(w, threads))
    run(ws[0])                                                    # warm-up (thread pool, plan tables)
    reps, t0 = 0, time.perf_counter()
    while True:
        run(ws[reps % 4])
        reps += 1
        el = time.perf_counter() - t0
        if el >= min_seconds and reps >= 2:
            break
    return reps * n_corr * 1024 / el, "%d corridors x 1024 pairs of the cfg4 fixture per pass, %d passes, %.1f s" % (n_corr, reps, el)


def reference_code_setup_ms():
    """What the REFERENCE'S OWN solverGurobi.cpp (compiled from /root/reference over a recording Gurobi stand-in,
    oracle/_ref/libsolver_ref.so: it travels to the GPU box prebuilt) spends per trial on model set-up alone, single core, no solve:
    a lower bound on the reference's cost per time-allocation factor (one trial = all assignments of one (corridor, dt))."""
    try:
        from oracle import solver_ref as sr
        if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libsolver_ref.so")):
            return None
        w = load_cfg4(0, 1)
        out = {}
        fd, saved = os.open(os.devnull, os.O_WRONLY), os.dup(1)   # the reference prints from its constructor
        os.dup2(fd, 1)
        try:
            for kind, N, ff in (("whole", w["N_whole"], True), ("safe", w["N_safe"], False)):
                po_, fo, Ab = w["poly_ofs_" + kind], w["face_ofs_" + kind], w["Ab_" + kind]
                polys = [(Ab[fo[q]:fo[q + 1], :3], Ab[fo[q]:fo[q + 1], 3]) for q in range(po_[0], po_[1])]
                x0 = w["x0"][0] if kind == "whole" else w["R_oracle"][0]
                sr.time_setup(N, x0, w["xf_" + kind][0], w["lim"][0], polys, ff, w["DC"], 3)
                out[kind] = 1e3 * sr.time_setup(N, x0, w["xf_" + kind][0], w["lim"][0], polys, ff, w["DC"], 20)
        finally:
            try:
                import ctypes
                ctypes.CDLL(None).fflush(None)                    # whatever the C++ side still buffers goes to /dev/null too
            except Exception:
                pass
            os.dup2(saved, 1)
            os.close(fd)
            os.close(saved)
        out["what"] = ("ms per trial of the reference's own createVars/set*Constraints/setObjective code (solverGurobi.cpp:445-455 without "
                       "optimize()), one core, Gurobi objects replaced by a recording stand-in: a lower bound; one trial covers the "
                       "%d / %d assignments of one (corridor, time allocation)" % (len(w["sigmas_whole"]), len(w["sigmas_safe"])))
        return out
    except Exception as e:
        return {"error": repr(e)[:160]}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path cannot run (Gurobi is closed source and
    absent); this times the tuned CPU port of the path (oracle/fq_cpu_port.c driving the chain of oracle/pair_oracle.py) on
    all host threads: same workload (the committed cfg4 fixture), a bounded sample per step.  Loads neither the product
    library nor a GPU."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    from oracle import pyoracle as po, pair_oracle
    po.build()
    n_s = max(1, args.ref_corridors)
    ws = [load_cfg4(256 + n_s * k, n_s) for k in range(4)]
    for k in range(max(1, args.warmup)):
        po.replan_pairs_port(ws[k % 4], threads)
    step_s = []
    for k in range(args.steps):
        t0 = time.perf_counter()
        po.replan_pairs_port(ws[k % 4], threads)                  # the whole chain in C (fqc_replan_pairs)
        step_s.append(time.perf_counter() - t0)
    el = float(sum(step_s))
    value = args.steps * n_s * 1024 / el
    # the literal restatement (the checker) beside it, for the record
    wl = load_cfg4(256, max(1, n_s // 8))
    t0 = time.perf_counter()
    pair_oracle.replan_pairs(wl, threads, fast=False)
    lit = wl["n_prob"] * 1024 / (time.perf_counter() - t0)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg4_config(args.gpus, args.corridors),
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port",
                             "sample": "%d corridors x 1024 pairs of the cfg4 fixture per step" % n_s, "note": CPU_NOTE,
                             "step_ms_p50_p99": [float(np.percentile(step_s, 50) * 1e3), float(np.percentile(step_s, 99) * 1e3)],
                             "literal_restatement_pairs_per_s": lit, "os_cpu_count": os.cpu_count(),
                             "reference_code_setup_ms_per_trial": reference_code_setup_ms()},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
class PairBatch:
    """One batch of corridors resident on the device + its output arrays, and the PairArgs pointing at them."""

    def __init__(self, w, dev, torch, capi, gather_world=0):
        self.w = w
        self.d = {k: torch.from_numpy(np.ascontiguousarray(w[k])).to(dev) for k in PAIR_KEYS}
        n, nc = w["n_prob"], pairs_per_pass(w)
        self.out = dict(feasible_whole=torch.zeros(nc, dtype=torch.uint8, device=dev), cost_whole=torch.zeros(nc, dtype=torch.float64, device=dev),
                        feasible_safe=torch.zeros(nc, dtype=torch.uint8, device=dev), cost_safe=torch.zeros(nc, dtype=torch.float64, device=dev),
                        results=torch.zeros(n * 144, dtype=torch.uint8, device=dev))
        self.gathered = torch.zeros(max(1, gather_world) * n * 144, dtype=torch.uint8, device=dev) if gather_world else None
        self.args = capi.pair_args(w, lambda k: self.d[k].data_ptr(), {k: v.data_ptr() for k, v in self.out.items()})

    def results(self, capi):
        return np.frombuffer(self.out["results"].cpu().numpy().tobytes(), capi.PAIR_RESULT_DTYPE)


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes path/<name>.npy for each array: 0/1 flags as float32, everything else as float64.  Above DUMP_BYTES in all, every
    array keeps the same seeded sample of its rows (the same rows for the same length), so two runs with the same arguments
    stay comparable entry for entry.  Every value written is finite: a value that is not is refused."""
    arrays = {k: np.asarray(v, np.float32 if v.dtype == np.uint8 else np.float64) for k, v in arrays.items()}
    for k, v in arrays.items():
        if not np.isfinite(v).all():
            raise ValueError("output %s has %d non-finite entries" % (k, int((~np.isfinite(v)).sum())))
    keep = min(1.0, DUMP_BYTES / sum(v.nbytes for v in arrays.values()))
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        if keep < 1.0:
            n = len(v)
            v = v[np.sort(np.random.default_rng(0).choice(n, max(1, int(n * keep)), replace=False))]
        np.save(os.path.join(path, k + ".npy"), v)


def pair_outputs(batches, capi):
    """What fq_replan_pairs_dev hands its caller, batch after batch: per-candidate flags and costs of both sweeps, and the
    fields of the per-corridor result records.  Where the library reports no result (include/faster_b200.h: the cost of a
    candidate its flag marks infeasible; the cost and dt of a sweep without a winner, whose dt index is -1; R, and the safe
    sweep's dt base, when the whole sweep has no winner) it leaves inf or nan: those entries are written as 0, the flags and
    indices beside them say which they are."""
    out = {k: np.concatenate([b.out[k].cpu().numpy() for b in batches])
           for k in ("feasible_whole", "cost_whole", "feasible_safe", "cost_safe")}
    res = np.concatenate([b.results(capi) for b in batches])
    out.update({"result_" + f: res[f] for f in capi.PAIR_RESULT_DTYPE.names})
    for s in ("whole", "safe"):
        out["cost_" + s] = np.where(out["feasible_" + s] != 0, out["cost_" + s], 0.0)
        won = res[s + "_dt_index"] >= 0
        for f in (s + "_cost", s + "_dt"):
            out["result_" + f] = np.where(won, res[f], 0.0)
    whole_won = res["whole_dt_index"] >= 0
    out["result_R"] = np.where(whole_won[:, None], res["R"], 0.0)
    out["result_safe_dt_base"] = np.where(whole_won, res["safe_dt_base"], 0.0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg4", choices=["cfg4", "cfg2", "cfg3", "cfg5"])
    ap.add_argument("--corridors", type=int, default=64, help="corridors per GPU per pass (cfg4)")
    ap.add_argument("--inner", type=int, default=64, help="passes per step")
    ap.add_argument("--ring", type=int, default=8, help="distinct batches a step cycles through")
    ap.add_argument("--ref-corridors", type=int, default=64, help="corridors per step of the CPU arm (the same 64 as one GPU pass)")
    ap.add_argument("--cpu-seconds", type=float, default=6.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--single-stream", action="store_true", help="all chains on one stream / context (no overlap of consecutive batches)")
    ap.add_argument("--contexts", type=int, default=3, help="solver contexts / streams the chains of consecutive batches rotate over")
    ap.add_argument("--quick", action="store_true", help="profiling runs: main timing only")
    ap.add_argument("--no-memo", action="store_true", help="A/B: switch the infeasibility-certificate memo off (option cert_memo = 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed as DIR/<name>.npy "
                                                          "(rank 0; at most 64 MB, a fixed seeded sample of larger outputs; entries without a "
                                                          "result, as the flags and indices show, are 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from faster_b200 import capi
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.config != "cfg4":
        line = bench_single(args, args.config, torch, capi, dev, local, world, rank, barrier, main_line=True)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- contexts: two (chains of consecutive batches overlap on two streams), each attached to the communicator
    n_ctx = 1 if args.single_stream else max(1, args.contexts)
    solvers = [capi.Solver(local) for _ in range(n_ctx)]
    if args.no_memo:
        for sv in solvers:
            sv.set_option("cert_memo", 0)
    if world > 1:
        for k, sv in enumerate(solvers):                     # one communicator per context: collectives of the two streams
            uid = [capi.comm_unique_id() if rank == 0 else None]      # must not share one (NCCL orders per communicator)
            dist.broadcast_object_list(uid, src=0)
            sv.comm_init(uid[0], rank, world)
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_ctx)]
    tstream = torch.cuda.Stream(device=dev)                  # timing stream: forks to / joins from the chain streams
    torch.cuda.set_stream(tstream)
    C, ring, inner = args.corridors, args.ring, args.inner
    ring = ((ring + n_ctx - 1) // n_ctx) * n_ctx            # a batch always meets the same context / stream
    n_fix = 512
    batches = [PairBatch(load_cfg4(((rank * ring + b) * C) % n_fix, C), dev, torch, capi, gather_world=world if world > 1 else 0)
               for b in range(ring)]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    ev_fork = torch.cuda.Event()
    ev_join = [torch.cuda.Event() for _ in range(max(n_ctx, STRONG_CONTEXTS))]

    def run_passes(n_pass, bl, sv=None, st=None):
        sv, st = sv or solvers, st or streams
        ev_fork.record(tstream)
        for s in st:
            s.wait_event(ev_fork)
        for p in range(n_pass):
            k = p % len(sv)
            b = bl[p % len(bl)]
            sv[k].replan_pairs_dev(b.args, b.gathered.data_ptr() if b.gathered is not None else 0, st[k].cuda_stream)
        for k, s in enumerate(st):
            ev_join[k].record(s)
            tstream.wait_event(ev_join[k])

    def timed(n_steps, n_pass, bl, sv=None, st=None):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        barrier()
        for i in range(n_steps):
            flush.zero_()                                    # L2 flush between timed steps (outside the events)
            ev[i][0].record(tstream)
            run_passes(n_pass, bl, sv, st)
            ev[i][1].record(tstream)
        barrier()
        return [a.elapsed_time(b) for a, b in ev]

    for _ in range(args.warmup):
        run_passes(inner, batches)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    step_ms = timed(args.steps, inner, batches)
    total_ms = float(sum(step_ms))
    res0 = batches[0].results(capi)
    if args.dump_outputs and rank == 0:                      # the batches the last step's passes wrote, before later legs reuse them
        dump_outputs(args.dump_outputs, pair_outputs(batches[:min(inner, len(batches))], capi))

    # ---- strong scaling: the SAME 64 corridors x 1024 pairs split over the ranks (cfg4 as written: 65 536 over 8 GPUs)
    strong = None
    if world > 1:
        lo, hi = capi.shard_range(C, None, rank, world)
        # a shard of 8-32 corridors does not fill the GPU: more chains in flight (measured on one GPU, 8 corridors per pass:
        # 21 / 49 / 58 M pairs/s with 1 / 3 / 6 contexts; profiles/r02p_contexts.log), each with its own communicator
        n_s = n_ctx if args.single_stream else max(n_ctx, STRONG_CONTEXTS)
        sv_s, st_s = list(solvers), list(streams)
        for k in range(n_ctx, n_s):
            sv = capi.Solver(local)
            uid = [capi.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            sv.comm_init(uid[0], rank, world)
            sv_s.append(sv)
            st_s.append(torch.cuda.Stream(device=dev))
        ring_s = ((ring + n_s - 1) // n_s) * n_s
        sb = [PairBatch(load_cfg4((b * C + lo) % n_fix, hi - lo), dev, torch, capi, gather_world=world) for b in range(ring_s)]
        # equal shard sizes are what the all-gather needs: C is a multiple of the world sizes used (64 / 2,4,8)
        run_passes(inner, sb, sv_s, st_s)
        sms = timed(max(3, args.steps // 2), inner, sb, sv_s, st_s)
        t = torch.tensor([float(sum(sms))], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong = {"scaling": "strong", "value": C * 1024 * inner * len(sms) / (float(t.item()) * 1e-3), "unit": "pairs/s",
                  "pairs_per_pass_total": C * 1024, "corridors_per_gpu_per_pass": hi - lo, "steps": len(sms), "contexts": n_s}
        del sb

    # ---- e2e: pinned host arrays through fq_replan_pairs_async, two contexts alternating
    host = []
    for b in batches[:max(3, n_ctx)]:
        hw = dict(b.w)
        for k in PAIR_KEYS:
            hw[k] = torch.from_numpy(np.ascontiguousarray(b.w[k])).pin_memory().numpy()
        n, nc = hw["n_prob"], pairs_per_pass(hw)
        ho = dict(results=torch.zeros(n * 144, dtype=torch.uint8).pin_memory().numpy().view(capi.PAIR_RESULT_DTYPE),
                  feasible_whole=torch.zeros(nc, dtype=torch.uint8).pin_memory().numpy(), cost_whole=torch.zeros(nc, dtype=torch.float64).pin_memory().numpy(),
                  feasible_safe=torch.zeros(nc, dtype=torch.uint8).pin_memory().numpy(), cost_safe=torch.zeros(nc, dtype=torch.float64).pin_memory().numpy())
        host.append((hw, ho))
    e2e_solvers = [capi.Solver(local) for _ in range(max(2, n_ctx))]     # plain contexts: the e2e leg measures the host path of one GPU
    if args.no_memo:
        for sv in e2e_solvers:
            sv.set_option("cert_memo", 0)

    def e2e_passes(n_pass):
        for p in range(n_pass):
            hw, ho = host[p % len(host)]
            e2e_solvers[p % len(e2e_solvers)].replan_pairs(hw, deferred=True, out=ho)
        for sv in e2e_solvers:
            sv.wait()
    e2e_inner = max(2, inner // 4)
    e2e_passes(4)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_passes(e2e_inner)
    barrier()
    e2e_s = time.perf_counter() - t0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    same = bool(host[0][1]["results"].tobytes() == res0.tobytes())
    h2d = sum(int(host[0][0][k].nbytes) for k in PAIR_KEYS)
    d2h = sum(int(v.nbytes) for v in host[0][1].values())

    t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_s = [float(x) for x in t.cpu()]
    pairs_pass = world * C * 1024
    value = pairs_pass * inner * args.steps / (total_ms * 1e-3)
    e2e = pairs_pass * e2e_inner * args.steps / e2e_s

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": cfg4_config(world, C),
                "run": {"passes_per_step": inner, "distinct_batches": ring, "certificate_memo": bool(capi.has_feature("cert_memo")) and not args.no_memo,
                        "streams": "one" if n_ctx == 1 else
                                   "%d contexts / streams: the chains of consecutive batches overlap (the tail of one fills with the next)" % n_ctx},
                "timed_region_s": total_ms * 1e-3,
                "step_ms": {"p50": float(np.percentile(step_ms, 50)), "p99": float(np.percentile(step_ms, 99)),
                            "min": float(np.min(step_ms)), "max": float(np.max(step_ms)), "note": "rank 0's steps"},
                "ms_per_pass": total_ms / args.steps / inner,
                "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": h2d * e2e_inner, "d2h_bytes_per_step": d2h * e2e_inner,
                        "passes_per_step": e2e_inner, "h2d_bytes_per_pass": h2d, "d2h_bytes_per_pass": d2h,
                        "how": "fq_replan_pairs_async on %d solver contexts + fq_wait; pinned host arrays; per-candidate flags and costs of both sweeps and the result records come back" % len(e2e_solvers),
                        "matches_resident": same},
                "gpu_launches": 11 * inner * args.steps,
                "gpu_launches_note": "per pass: 2 dt-base, 2 grid-expand, 2 sweep solves, 2 selections, 1 winners' solve, R sampling, result records",
                "clocks": sampler.summary()}
        if strong:
            line["strong"] = strong
    if args.quick:
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- the dominant kernel alone: the two sweep launches of batch 0, replicated on expanded arrays, CUDA-event timed
    kern = sweep_kernel_times(batches[0], res0, e2e_solvers[0], torch, capi, dev, tstream, flush)
    # one chain alone on one stream (no overlap with a neighbouring batch), same cold-cache conditions as the kernel timing:
    # the denominator of the sweep kernels' share of a pass (to be compared with the serialised ncu launch list)
    serial = []
    for _ in range(10):
        flush.zero_()
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(tstream)
        solvers[0].replan_pairs_dev(batches[0].args, batches[0].gathered.data_ptr() if batches[0].gathered is not None else 0, tstream.cuda_stream)
        z.record(tstream)
        torch.cuda.synchronize()
        serial.append(a.elapsed_time(z))
    serial_pass_ms = float(np.mean(serial[2:]))
    if rank == 0:
        feas = np.concatenate([batches[0].out["feasible_whole"].cpu().numpy(), batches[0].out["feasible_safe"].cpu().numpy()])
        line["config"]["feasible_fraction"] = float(feas.mean())
        line["config"]["mean_active_set_iters"] = kern["mean_iters"]
        line["config"]["active_set_iters_p99_max"] = kern["iters_p99_max"]
        line["config"]["iteration_cap_hits"] = kern["cap_hits"]
        nc = C * 1024
        kernel_ms = 0.5 * (kern["whole_ms"] + kern["safe_ms"])
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = nc * BYTES_PER_CAND[10] / (kernel_ms * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": None, "kernel": "fqt::fq_solve_kernel_t<10,*> (whole and safe sweep launches)",
                            "kernel_ms": kernel_ms, "kernel_ms_whole": kern["whole_ms"], "kernel_ms_safe": kern["safe_ms"],
                            "serial_pass_ms": serial_pass_ms,
                            "kernel_share_of_pass": (kern["whole_ms"] + kern["safe_ms"]) / serial_pass_ms,
                            "kernel_share_note": "the two sweep launches over one chain run alone on one stream (the timed region overlaps "
                                                 "%d chains, so its ms_per_pass is below the serial pass time); the ncu launch list of the "
                                                 "same chain gives 92 %% (profiles/)" % n_ctx,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s",
                            "algorithmic_bytes_per_candidate": BYTES_PER_CAND[10],
                            "note": "HBM fraction is tiny by construction (SURVEY 8d: 195 B and ~4 k warp instructions per candidate); "
                                    "the nearest hardware limits are the shared-memory data pipe and issue slots: see ncu"}
        line["roofline"].update(ncu_summary(kernel_ms, nc, float(line["clocks"].get("sm_mhz") or 0.0)))
    # ---- parity: a slice of batch 0 against the CPU restatement of the chain, and the tolerance / margin picture
    if rank == 0 and not args.no_cpu_baseline:
        line["parity"] = parity_block(batches[0], res0, e2e_solvers[0], torch, capi, dev)
    # ---- what a planner needs from a replan is the WINNERS (first feasible factor, then minimum cost): with the library's
    #      early exit (option "sweep_early_exit") candidates that cannot win are not evaluated.  Not the BASELINE metric
    #      (those candidates are not solved); reported as replans (corridor pairs) per second beside the full evaluation.
    if rank == 0:
        ee = capi.Solver(local)
        ee.set_option("sweep_early_exit", 1)
        rates = {}
        for name, sv in (("full_evaluation", e2e_solvers[0]), ("early_exit", ee)):
            for _ in range(3):
                sv.replan_pairs_dev(batches[0].args, 0, tstream.cuda_stream)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(tstream)
            for p in range(inner):
                sv.replan_pairs_dev(batches[p % ring].args, 0, tstream.cuda_stream)
            a1.record(tstream)
            torch.cuda.synchronize()
            rates[name] = C * inner / (a0.elapsed_time(a1) * 1e-3)
            if name == "early_exit":
                res_ee = batches[(inner - 1) % ring].results(capi)
        sv = e2e_solvers[0]
        sv.replan_pairs_dev(batches[(inner - 1) % ring].args, 0, tstream.cuda_stream)
        torch.cuda.synchronize()
        res_full = batches[(inner - 1) % ring].results(capi)
        line["replans_per_s"] = {"full_evaluation": rates["full_evaluation"], "early_exit": rates["early_exit"], "unit": "corridor pairs/s",
                                 "how": "fq_replan_pairs_dev, one context / stream, %d corridors per pass" % C,
                                 "same_winners": bool(res_ee.tobytes() == res_full.tobytes())}
        ee.close()
    # ---- single-replan latency (what the robot experiences against its 10 ms budget)
    if rank == 0:
        line["replan_latency_us"] = latency_block(e2e_solvers[0], capi)
    if rank == 0 and not args.no_cpu_baseline:
        threads = host_threads()
        rate, sample = cpu_pair_rate(args.ref_corridors, threads, args.cpu_seconds)
        lit, _ = cpu_pair_rate(max(1, args.ref_corridors // 8), threads, 2.0, fast=False)
        line["cpu_baseline"] = {"value": rate, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": sample,
                                "note": CPU_NOTE, "literal_restatement_pairs_per_s": lit, "os_cpu_count": os.cpu_count()}
        # (the reference code's own set-up time per trial is measured in the `--impl reference` arm's line, which loads no GPU)
    if world == 1 and not args.no_other_configs:
        line["other_configs"] = {}
        for name in ("cfg2", "cfg3", "cfg5"):
            try:
                line["other_configs"][name] = bench_single(args, name, torch, capi, dev, local, world, rank, barrier, main_line=False)
            except Exception as e:                        # a side measurement must not take the main line down
                line["other_configs"][name] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def ncu_summary(kernel_ms, n_cand=0, sm_mhz=0.0):
    """DRAM traffic and pipe utilisation come from the committed ncu capture of this kernel (profiles/): they cannot be
    measured inside an unprofiled run."""
    try:
        pj = json.load(open(os.path.join(ROOT, "profiles", "kernel_metrics_latest.json")))
        ls = [l for l in pj["launches"] if "fq_solve_kernel" in l["kernel"] and int(l["grid"].strip("()").split(",")[0]) >= 148]
        out = {"traffic": float(np.mean([l["dram_bytes"] for l in ls])),
               "ncu": {"source": pj["label"], "fp64_pipe_active_pct": float(np.mean([l["fp64_pipe_active_pct"] for l in ls])),
                       "issue_active_pct": float(np.mean([l["issue_active_pct"] for l in ls]))}}
        if all("lsu_data_pipe_pct_of_peak" in l for l in ls):
            out["ncu"]["shared_memory_pipe_pct_of_peak"] = float(np.mean([l["lsu_data_pipe_pct_of_peak"] for l in ls]))
        if all("fp64_flop" in l for l in ls) and n_cand and sm_mhz:
            # SURVEY 8(d)'s second roofline: fp64 flops the kernel executes (ncu's thread-level DFMA x2 + DADD + DMUL of
            # the same launches, per candidate) x the live candidate rate, against the DFMA peak at the live SM clock
            per_cand = float(np.mean([l["fp64_flop"] for l in ls])) / 65536.0
            peak = float(ls[0]["fp64_peak_flop_per_cycle"]) * sm_mhz * 1e6 / 1e12
            ach = per_cand * n_cand / (kernel_ms * 1e-3) / 1e12
            out["fp64"] = {"flop_per_candidate": per_cand, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                           "peak_source": "ncu DFMA peak_sustained (%d flop/cycle over the chip) x SM clock under load" % int(ls[0]["fp64_peak_flop_per_cycle"])}
        return out
    except Exception:
        return {}


def expanded_arrays(b, res, kind, torch, dev):
    """The candidate arrays the chain builds on the device, rebuilt from the result records (dt bases, R): lets the sweep
    launches run alone through fq_solve_multi_dev and the oracle check exactly the same candidates."""
    w = b.w
    n = w["n_prob"]
    fac, sig = w["factors_" + kind], w["sigmas_" + kind]
    base = res["whole_dt_base" if kind == "whole" else "safe_dt_base"]
    dts = (base[:, None, None] * fac[None, :, None] * np.ones((1, 1, len(sig)))).reshape(-1)
    sg = np.ascontiguousarray(np.broadcast_to(sig[None, None], (n, len(fac), len(sig), sig.shape[1])).reshape(-1, sig.shape[1]))
    co = (np.arange(n + 1) * len(fac) * len(sig)).astype(np.int32)
    x0 = w["x0"] if kind == "whole" else np.ascontiguousarray(res["R"])
    return dict(x0=x0, xf=w["xf_" + kind], dt=np.ascontiguousarray(dts), sigma=sg, cand_ofs=co)


def sweep_kernel_times(b, res, solver, torch, capi, dev, tstream, flush):
    out = {}
    iters_all = []
    for kind, N, ff in (("whole", b.w["N_whole"], True), ("safe", b.w["N_safe"], False)):
        e = expanded_arrays(b, res, kind, torch, dev)
        d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in e.items()}
        nc = len(e["dt"])
        feas = torch.zeros(nc, dtype=torch.uint8, device=dev); cost = torch.zeros(nc, dtype=torch.float64, device=dev)
        its = torch.zeros(nc, dtype=torch.int32, device=dev)
        solver.set_option("max_faces_per_polytope", b.w["max_poly_faces_" + kind])

        def launch(with_iters):
            solver.solve_multi_dev(N, ff, b.w["n_prob"], d["x0"].data_ptr(), d["xf"].data_ptr(), b.d["lim"].data_ptr(),
                                   b.d["poly_ofs_" + kind].data_ptr(), b.d["face_ofs_" + kind].data_ptr(), b.d["Ab_" + kind].data_ptr(),
                                   d["cand_ofs"].data_ptr(), nc // b.w["n_prob"], b.w["max_faces_" + kind], d["dt"].data_ptr(),
                                   d["sigma"].data_ptr(), feas.data_ptr(), cost.data_ptr(), 0, its.data_ptr() if with_iters else 0,
                                   tstream.cuda_stream)
        launch(False)
        ms = []
        for _ in range(10):
            flush.zero_()
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(tstream); launch(False); z.record(tstream)
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(z))
        out[kind + "_ms"] = float(np.mean(ms))
        launch(True)
        torch.cuda.synchronize()
        assert bool(torch.equal(feas, b.out["feasible_" + kind])), "replicated %s sweep differs from the chain's" % kind
        iters_all.append(its.cpu().numpy())
    solver.set_option("max_faces_per_polytope", 0)
    it = np.concatenate(iters_all)
    out["cap_hits"] = int((it < 0).sum())
    it = np.abs(it).astype(float)
    out["mean_iters"] = float(it.mean())
    out["iters_p99_max"] = [float(np.percentile(it, 99)), float(it.max())]
    return out


def parity_block(b, res, solver, torch, capi, dev, n_chk=4):
    """Oracle check of the first corridors of batch 0, plus what the row tolerance does to the flags."""
    from oracle import pair_oracle, pyoracle as po
    w = load_cfg4_like(b.w, n_chk)
    g = solver.replan_pairs(w)
    r = g["results"]
    o = pair_oracle.replan_pairs(w, os.cpu_count() or 1, dt_base_whole=r["whole_dt_base"], dt_base_safe=r["safe_dt_base"])
    mism = int((g["feasible_whole"] != o["feasible_whole"]).sum() + (g["feasible_safe"] != o["feasible_safe"]).sum())
    worst = 0.0
    for k in ("whole", "safe"):
        ok = o["feasible_" + k].astype(bool) & g["feasible_" + k].astype(bool)
        if ok.any():
            worst = max(worst, float((np.abs(g["cost_" + k][ok] - o["cost_" + k][ok]) / np.maximum(1e-9, np.abs(o["cost_" + k][ok]))).max()))
    out = {"checked_candidates": int(2 * pairs_per_pass(w)), "flag_mismatches": mism, "max_rel_cost_err": worst,
           "winner_mismatches": int((r["whole_dt_index"] != o["whole_dt_index"]).sum() + (r["whole_sigma_index"] != o["whole_sigma_index"]).sum() +
                                    (r["safe_dt_index"] != o["safe_dt_index"]).sum() + (r["safe_sigma_index"] != o["safe_sigma_index"]).sum()),
           "dt_base_mismatches_device_vs_cpu": int((r["whole_dt_base"] != o["whole_dt_base_own"]).sum()),
           "against": "oracle/ (CPU restatement of the chain), same inputs"}
    # tolerance regime: Gurobi's default FeasibilityTol is 1e-6 (the reference sets none, solverGurobi.cpp:479-487); ours 1e-8
    full = b.w
    base = solver.replan_pairs(full, want_coeffs=False)
    solver.set_option("row_tol_1e9", 1000)
    loose = solver.replan_pairs(full, want_coeffs=False)
    solver.set_option("row_tol_1e9", 10)
    flips = {k: int((base["feasible_" + k] != loose["feasible_" + k]).sum()) for k in ("whole", "safe")}
    out["flag_flips_tol_1e-6_vs_1e-8"] = {"whole": flips["whole"], "safe": flips["safe"], "of": int(pairs_per_pass(full)),
                                          "winner_changes": int((base["results"]["whole_dt_index"] != loose["results"]["whole_dt_index"]).sum() +
                                                                (base["results"]["safe_dt_index"] != loose["results"]["safe_dt_index"]).sum())}
    # feasibility margins: flags with every polytope offset b and every limit moved by s (s < 0 tightens).  A candidate
    # whose flag differs between -s and +s lies within s of the feasibility boundary.
    hist = {}
    for s in (1e-6, 1e-5, 1e-4, 1e-3):
        fl = []
        for sign in (-1.0, 1.0):
            ws = dict(full)
            for k in ("whole", "safe"):
                A = full["Ab_" + k].copy(); A[:, 3] += sign * s; ws["Ab_" + k] = A
            ws["lim"] = full["lim"] + sign * s
            fl.append(solver.replan_pairs(ws, want_coeffs=False))
        hist["within_%g" % s] = {k: int((fl[0]["feasible_" + k] != fl[1]["feasible_" + k]).sum()) for k in ("whole", "safe")}
    out["feasibility_margin_counts"] = hist
    out["feasibility_margin_note"] = "candidates whose flag changes when every row bound moves by -s vs +s (m, m/s, m/s2, m/s3); safe counts include the effect on R"
    out["proved_on_literal_model"] = proof_sample(full, base["results"], solver)
    return out


def proof_sample(w, rr, solver, n_corr=2, n_cand=24):
    """A sample of the batch's candidates PROVED on the literal rows of the reference's model (oracle/proofs.py, checker only):
    "solved" -> the GPU's coefficients are feasible there and carry KKT multipliers (optimal); "not solved" -> the Farkas
    certificate exported by fq_solve_batch_cert holds.  No solver's verdict enters.  tools/stress_proofs.py is the large run."""
    out = {"candidates": 0, "solved_proved_optimal": 0, "not_solved_proved_infeasible": 0, "without_proof": 0, "failures": 0}
    try:
        from oracle import model_fullspace as mf, proofs
        rng = np.random.default_rng(4)
        for j in range(min(n_corr, w["n_prob"])):
            for kind, N, ff in (("whole", w["N_whole"], True), ("safe", w["N_safe"], False)):
                base = rr[kind + "_dt_base"][j]
                x0 = w["x0"][j] if kind == "whole" else rr["R"][j]
                if not np.isfinite(base) or not np.all(np.isfinite(x0)):
                    continue
                po_, fo, Ab = w["poly_ofs_" + kind], w["face_ofs_" + kind], w["Ab_" + kind]
                polys = [(Ab[fo[q]:fo[q + 1], :3].copy(), Ab[fo[q]:fo[q + 1], 3].copy()) for q in range(po_[j], po_[j + 1])]
                fac, sig = w["factors_" + kind], w["sigmas_" + kind]
                dts = fac[rng.integers(0, len(fac), n_cand)] * base
                sigs = sig[rng.integers(0, len(sig), n_cand)]
                fg, cg, cog, _ = solver.solve_batch(N, x0, w["xf_" + kind][j], w["lim"][j], polys, dts, sigs, ff, want_coeffs=True)
                fc, _, cert = solver.solve_batch_cert(N, x0, w["xf_" + kind][j], w["lim"][j], polys, dts, sigs, ff)
                for i in range(n_cand):
                    out["candidates"] += 1
                    model = mf.build(N, x0, w["xf_" + kind][j], w["lim"][j], dts[i], polys, sigs[i], ff)
                    try:
                        if fg[i] != fc[i]:
                            raise AssertionError("kernels disagree")
                        if fg[i]:
                            proofs.assert_optimal(model, cog[i], cg[i]); out["solved_proved_optimal"] += 1
                        elif int(cert[i, 0]) >= 1:
                            proofs.assert_infeasible(model, N, polys, sigs[i], cert[i]); out["not_solved_proved_infeasible"] += 1
                        else:
                            out["without_proof"] += 1
                    except AssertionError:
                        out["failures"] += 1
    except Exception as e:                                    # the checker must never take the measurement down
        out["error"] = repr(e)[:200]
    return out


def load_cfg4_like(w, n):
    """First n corridors of a pair workload dict."""
    out = dict(w)
    out["n_prob"] = n
    for k in ("x0", "xf_whole", "xf_safe", "lim"):
        out[k] = np.ascontiguousarray(w[k][:n])
    for kind in ("whole", "safe"):
        po, fo = w["poly_ofs_" + kind], w["face_ofs_" + kind]
        out["poly_ofs_" + kind] = np.ascontiguousarray(po[:n + 1])
        out["face_ofs_" + kind] = np.ascontiguousarray(fo[:po[n] + 1])
        out["Ab_" + kind] = np.ascontiguousarray(w["Ab_" + kind][:fo[po[n]]])
    return out


def latency_block(solver, capi):
    from faster_b200 import corridor as cr
    w = load_cfg4(0, 1)
    polys = [(w["Ab_whole"][w["face_ofs_whole"][p]:w["face_ofs_whole"][p + 1], :3], w["Ab_whole"][w["face_ofs_whole"][p]:w["face_ofs_whole"][p + 1], 3])
             for p in range(3)]
    x0, xf, lim = w["x0"][0], w["xf_whole"][0], w["lim"][0]
    sig66 = cr.monotone_sigmas(N_SEG, 3)
    dts10 = np.arange(1.0, 11.0) * max(capi.dt_initial(x0, xf, lim, N_SEG), 0.02)

    def med(fn, n=50, skip=10):
        lat = []
        for _ in range(n):
            t0 = time.perf_counter(); r = fn(); lat.append(time.perf_counter() - t0)
        return float(np.median(lat[skip:]) * 1e6), r
    def med2(fn, n=50, skip=10):
        """the same call with the early exit off / on, ALTERNATING (clock ramps and host noise hit both alike)"""
        lat = ([], [])
        r = [None, None]
        for i in range(2 * n):
            solver.set_option("sweep_early_exit", i & 1)
            t0 = time.perf_counter(); r[i & 1] = fn(); lat[i & 1].append(time.perf_counter() - t0)
        solver.set_option("sweep_early_exit", 0)
        return float(np.median(lat[0][skip:]) * 1e6), r[0], float(np.median(lat[1][skip:]) * 1e6), r[1]
    w1 = load_cfg4(0, 1)
    # early exit = what the drop-in class does (include/solverGurobi.hpp switches it on: only the winner is needed)
    us, g, us_ee, g_ee = med2(lambda: solver.gen_new_traj(N_SEG, x0, xf, lim, polys, dts10, sig66, True))
    us_x, ge, us_x_ee, ge_ee = med2(lambda: solver.gen_new_traj_exact(N_SEG, x0, xf, lim, polys, dts10, True), 40)
    us_pair, rp, us_pair_ee, rp_ee = med2(lambda: solver.replan_pairs(w1, want_candidates=False), 40)
    import itertools
    pb6 = cr.make_corridor(10000, 3, 6)
    sig729 = np.array(list(itertools.product(range(3), repeat=6)), np.uint8)
    dts6 = np.arange(1.0, 11.0) * max(capi.dt_initial(pb6["x0"], pb6["xf"], pb6["lim"], 6), 2 * pb6["DC"])
    us6, _ = med(lambda: solver.gen_new_traj(6, pb6["x0"], pb6["xf"], pb6["lim"], pb6["polys"], dts6, sig729, True), 40)
    out = {"value": us, "what": "fq_gen_new_traj: 10 factors x 66 assignments, N=10, P=3 (a cfg4 forest corridor), host in/out, median",
           "exact_miqp": us_x, "exact_nodes": int(ge["nodes"]),
           "exact_same_winner": bool(ge["dt_index"] == g["dt_index"] and abs(ge["cost"] - g["cost"]) <= 1e-9 * max(1.0, g["cost"])),
           "early_exit": {"value": us_ee, "exact_miqp": us_x_ee, "chained_pair_one_corridor": us_pair_ee,
                          "same_winners": bool(g_ee["dt_index"] == g["dt_index"] and g_ee["cost"] == g["cost"] and ge_ee["cost"] == ge["cost"] and
                                               rp_ee["results"].tobytes() == rp["results"].tobytes()),
                          "what": "option sweep_early_exit = 1 (the drop-in class's setting): factors beyond the first feasible one are not evaluated"},
           "chained_pair_one_corridor": us_pair, "chained_pair_what": "fq_replan_pairs, 1 corridor: whole 16x64 -> R -> safe 16x64, winners' coefficients back",
           "shipped_yaml_N6_P3_all_729_assignments": us6}
    try:
        from oracle import pyoracle as po
        lat = []
        for _ in range(15):
            t0 = time.perf_counter()
            po.gen_new_traj(N_SEG, x0, xf, lim, polys, 0.01, 1.0, 10.0, 1.0, None, True)
            lat.append(time.perf_counter() - t0)
        out["cpu_restatement_exact_sweep"] = float(np.median(lat) * 1e6)
    except Exception:
        pass
    return out


def bench_single(args, name, torch, capi, dev, local, world, rank, barrier, main_line):
    """BASELINE configs 2 / 3 / 5: one kind of candidates, resident arrays, fq_solve_multi_dev."""
    cfg = SINGLE[name]
    C = cfg["corridors"]
    w = make_single(cfg, C, capi.dt_initial)
    keys = ["x0", "xf", "lim", "poly_ofs", "face_ofs", "Ab", "cand_ofs", "dt", "sigma"]
    d = {k: torch.from_numpy(np.ascontiguousarray(w[k])).to(dev) for k in keys}
    nc = C * w["cand"]
    feas = torch.zeros(nc, dtype=torch.uint8, device=dev); cost = torch.zeros(nc, dtype=torch.float64, device=dev)
    its = torch.zeros(nc, dtype=torch.int32, device=dev)
    solver = capi.Solver(local)
    solver.set_option("max_faces_per_polytope", w["max_poly_faces"])
    st = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(st)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def launch(n_prob=C, with_iters=False):
        solver.solve_multi_dev(w["N"], w["ff"], n_prob, d["x0"].data_ptr(), d["xf"].data_ptr(), d["lim"].data_ptr(),
                               d["poly_ofs"].data_ptr(), d["face_ofs"].data_ptr(), d["Ab"].data_ptr(), d["cand_ofs"].data_ptr(),
                               w["cand"], w["max_faces"], d["dt"].data_ptr(), d["sigma"].data_ptr(), feas.data_ptr(), cost.data_ptr(), 0,
                               its.data_ptr() if with_iters else 0, st.cuda_stream)
    per_launch_ms = None
    torch.cuda.synchronize()                             # the arrays above were filled on the previous current stream
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st); launch(); z.record(st); torch.cuda.synchronize()
    per_launch_ms = a.elapsed_time(z)
    inner = max(1, min(64, int(round((60.0 if main_line else 25.0) / max(per_launch_ms, 0.05)))))
    steps = args.steps if main_line else max(5, min(args.steps, 10))
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for i in range(steps):
        flush.zero_()
        ev[i][0].record(st)
        for _ in range(inner):
            launch()
        ev[i][1].record(st)
    barrier()
    if main_line and args.dump_outputs and rank == 0:
        f = feas.cpu().numpy()
        dump_outputs(args.dump_outputs, {"feasible": f, "cost": np.where(f != 0, cost.cpu().numpy(), 0.0)})   # as pair_outputs
    sms = [x.elapsed_time(y) for x, y in ev]
    total_ms = float(sum(sms))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    # single launches, L2 flushed: the kernel's own time; and the literal one-corridor batch of BASELINE
    kms, lit = [], []
    for _ in range(8):
        flush.zero_()
        a.record(st); launch(); z.record(st); torch.cuda.synchronize()
        kms.append(a.elapsed_time(z))
        a.record(st); launch(1); z.record(st); torch.cuda.synchronize()
        lit.append(a.elapsed_time(z))
    launch(with_iters=True)
    torch.cuda.synchronize()
    it = its.cpu().numpy()
    kernel_ms = float(np.mean(kms))
    value = world * nc * inner * steps / (total_ms * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    bpc = BYTES_PER_CAND[w["N"]]
    achieved = nc * bpc / (kernel_ms * 1e-3) / 1e9
    out = {"metric": "candidate trajectory solves/sec (single kind)", "value": value, "unit": "candidates/s", "n_gpus": world,
           "steps": steps, "warmup": 3, "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": cfg["name"], "corridors_per_gpu": C, "candidates_per_launch": nc, "launches_per_step": inner,
                      "l2": "flushed between timed steps", "feasible_fraction": float(feas.cpu().numpy().mean()),
                      "mean_active_set_iters": float(np.abs(it).mean()), "iteration_cap_hits": int((it < 0).sum())},
           "timed_region_s": total_ms * 1e-3, "gpu_launches": inner * steps,
           "literal_batch": {"what": "ONE corridor, %d candidates, one launch (BASELINE's batch as written): launch-latency bound" % w["cand"],
                             "ms": float(np.mean(lit)), "candidates_per_s": w["cand"] / (float(np.mean(lit)) * 1e-3)},
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                        "kernel": "fqt::fq_solve_kernel_t<%d,%d>" % (w["N"], 1 if w["ff"] else 0), "kernel_ms": kernel_ms,
                        "algorithmic_bytes_per_candidate": bpc, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s"}}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as po
        nchk = 1 if w["cand"] > 4096 else min(C, 4)
        ncand = nchk * w["cand"]
        sel = slice(0, ncand) if ncand <= 16384 else np.arange(0, ncand, ncand // 16384)
        fo, co = po.solve_multi(w["N"], w["ff"], w["x0"][:nchk], w["xf"][:nchk], w["lim"][:nchk], w["poly_ofs"][:nchk + 1],
                                w["face_ofs"][:w["poly_ofs"][nchk] + 1], w["Ab"][:w["face_ofs"][w["poly_ofs"][nchk]]],
                                w["cand_ofs"][:nchk + 1], w["dt"][:ncand], w["sigma"][:ncand], os.cpu_count() or 1)
        fg = feas[:ncand].cpu().numpy(); cg = cost[:ncand].cpu().numpy()
        ok = fo.astype(bool) & fg.astype(bool)
        out["parity"] = {"checked_candidates": int(ncand), "flag_mismatches": int((fg != fo).sum()),
                         "max_rel_cost_err": float((np.abs(cg[ok] - co[ok]) / np.maximum(1e-9, np.abs(co[ok]))).max()) if ok.any() else 0.0,
                         "against": "oracle/fq_oracle.c, same inputs"}
        nc_cpu = min(C, max(1, 65536 // w["cand"]))             # the tuned CPU port on about 65 536 candidates per pass
        sub = (w["N"], w["ff"], w["x0"][:nc_cpu], w["xf"][:nc_cpu], w["lim"][:nc_cpu], w["poly_ofs"][:nc_cpu + 1],
               w["face_ofs"][:w["poly_ofs"][nc_cpu] + 1], w["Ab"][:w["face_ofs"][w["poly_ofs"][nc_cpu]]], w["cand_ofs"][:nc_cpu + 1],
               w["dt"][:nc_cpu * w["cand"]], w["sigma"][:nc_cpu * w["cand"]], host_threads())
        fp, _ = po.solve_multi_port(*sub)
        out["parity"]["tuned_cpu_port_flag_mismatches_vs_gpu"] = int((fp != feas[:nc_cpu * w["cand"]].cpu().numpy()).sum())
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < (2.0 if not main_line else args.cpu_seconds):
            po.solve_multi_port(*sub)
            reps += 1
        out["cpu_baseline"] = {"value": reps * nc_cpu * w["cand"] / (time.perf_counter() - t0), "unit": "candidates/s", "cores": host_threads(),
                               "kind": "port", "sample": "%d corridor(s) x %d candidates, %d passes" % (nc_cpu, w["cand"], reps)}
    solver.close()
    return out


if __name__ == "__main__":
    main()
