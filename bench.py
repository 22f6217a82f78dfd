#!/usr/bin/env python
"""bench.py -- Monte-Carlo network evals/s (1 eval = one (sample, frequency) point).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg5] [--dump-outputs DIR]

Headline step = one pass of the hot path over one batch of synthetic input: BASELINE config 2
(pcb/generic-filter 11th-order 0.1 dB Chebyshev LPF with ESR/SRF parasitics, +-5 % L / +-2 % C,
1e6 tolerance samples x 4096 log-spaced frequency points, reduce-only yield + 256-bin histogram)
per GPU.  N > 1 (torchrun, one process per GPU) shards the samples: every rank takes 1e6 samples of
a global N x 1e6 job (weak scaling), and the only collective is the sum all-reduce of the uint64
counters.  Prints ONE JSON line (rank 0).

  value          whole-job evals/s with tables/grid/specs already resident in HBM (qo_plan_launch)
  e2e            the same through the host-buffer C-ABI call qo_mc_run (H2D of tables / specs / program and
                 D2H of the counters inside the timed region)
  roofline       EXECUTED FP64 flops of the dominant kernel (ncu instruction counts per eval, DFMA = 2, DMUL / DADD = 1;
                 profiles/executed_fp64.json) x the rate measured here, over the FP64-FMA peak MEASURED in this run by a
                 dependency-free DFMA loop (MEASURED_PEAKS.json holds no FP64 figure); alg_v1_ratio = the SURVEY 8d
                 algorithmic count over the same peak (> 1: the kernel does less work than ALG-v1 counts)
  north_star_job BASELINE config 5 -- coupled line + 11th-order ladder, 1e8 samples x 4096 points in TOTAL, sharded over the
                 N ranks (strong scaling): seconds for the job, evals/s, executed fraction, counters
  cpu_baseline / --impl reference
                 the CPU oracle (oracle/, the port of the models the reference's external tools apply) on the box's host
                 cores, on a bounded sample of the same workload, built WITHOUT the product library (oracle/ref_workloads.py)
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
sys.path.insert(0, ROOT)

REAL_STDOUT = sys.stdout
METRIC = "Monte Carlo network evals/s (samples x freq pts)"
UNIT = "evals/s"
SAMPLES_PER_GPU = 1000000
NF = 4096
NORTH_STAR_SAMPLES = 100000000          # BASELINE config 5: 1e8 samples x 4096 points
REF_SAMPLES_PER_STEP = 20000            # bounded sample of the reference arm (the workload is 1e6 per GPU per step)
# the polynomial (transfer-function) kernels: thread-per-sample for the bulk of a large launch, warp-per-sample for the rest
TF_KERNELS = ("qo_mc_ts_kernel", "qo_mc_tf_kernel")


def host_cores():
    """Cores this process may run on.  NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def kernel_source_hash():
    """sha256 over the kernel sources: profiles/executed_fp64.json records the hash its ncu captures were taken at."""
    d = os.path.join(ROOT, "qo-100-tools_b200", "csrc")
    h = hashlib.sha256()
    for n in sorted(os.listdir(d)):
        if n.endswith((".cu", ".cuh", ".h")):
            h.update(n.encode())
            h.update(open(os.path.join(d, n), "rb").read())
    return h.hexdigest()[:16]


def kernel_sass_hash(kernel):
    """hash of `kernel`'s machine code in the library being benchmarked (qo-100-tools_b200/lib/sass_hashes.json, written by
    build() from the object files the library was linked from), or None when the file is missing or describes another build of the library"""
    try:
        lib = os.path.join(ROOT, "qo-100-tools_b200", "lib")
        d = json.load(open(os.path.join(lib, "sass_hashes.json")))
        if d.get("lib_sha256") != hashlib.sha256(open(os.path.join(lib, "libqo100net.so"), "rb").read()).hexdigest():
            return None
        return d["kernels"][kernel]["sha"]
    except Exception:
        return None


def profile_match(ex, kernel):
    """Were the ncu counts taken on the code being benchmarked?  "source": same kernel sources; "sass": sources changed since, but
    this kernel's machine code is byte-identical to the profiled build's; False: neither."""
    if ex.get("src_hash") == kernel_source_hash():
        return "source"
    sh = kernel_sass_hash(kernel)
    return "sass" if sh is not None and sh == (ex.get("sass") or {}).get(kernel) else False


def executed_profile(plan_kernel, wl_name):
    """{"dfma", "dmul", "dadd" per eval, "dram_bytes_per_launch", "source", "src_hash"} of the kernel on this workload, or None."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "executed_fp64.json")))
        e = dict(d[plan_kernel]["cfg5" if wl_name.startswith("cfg5") else "cfg2"])
        e.setdefault("src_hash", d.get("_src_hash"))
        e.setdefault("git", d.get("_git"))
        e.setdefault("sass", d.get("_sass"))
        return e
    except Exception:
        return None


def executed_view(kernel, wl_name, evals_per_s_per_gpu, peak_tflops):
    """executed FP64 work of `kernel` (ncu counts per eval) at a measured per-GPU rate: tflops counts DFMA as 2; pipe_util =
    FP64-pipe instructions/s over the measured DFMA issue rate (peak TFLOP/s / 2)"""
    ex = executed_profile(kernel, wl_name)
    if not ex:
        return None
    ipe = ex["dfma"] + ex["dmul"] + ex["dadd"]
    fl = 2 * ex["dfma"] + ex["dmul"] + ex["dadd"]
    return {"flops_per_eval": fl, "fp64_pipe_instr_per_eval": ipe, "dfma_per_eval": ex["dfma"],
            "tflops": fl * evals_per_s_per_gpu * 1e-12, "frac_of_peak": fl * evals_per_s_per_gpu * 1e-12 / peak_tflops,
            "pipe_util": ipe * evals_per_s_per_gpu / (peak_tflops * 0.5e12),
            "ncu_fp64_pipe_active_pct": ex.get("fp64_pipe_active_pct"), "source": ex.get("source"), "profile_git": ex.get("git"),
            "profile_matches_source": bool(profile_match(ex, kernel)), "profile_match": profile_match(ex, kernel)}


def time_plan(plan, stream, counters, nspg, steps, warmup, torch):
    """mean kernel ms over `steps` launches of a resident plan (CUDA events on the launching stream)"""
    with torch.cuda.stream(stream):
        for i in range(warmup):
            plan.launch(i * nspg, nspg, counters.data_ptr())
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        for i in range(steps):
            plan.launch((warmup + i) * nspg, nspg, counters.data_ptr())
        b.record(stream)
        torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def workload(name, n_samples):
    from qo100net import workloads as W
    if name == "cfg5":
        return W.cfg5(n_samples, NF)
    return W.cfg2(n_samples, NF)


def cpu_reference(rwl, n_samples, steps, warmup, nthreads):
    """Times the oracle port (OpenMP over samples) on a bounded sample; returns (evals/s, s/step, counters of the last step)."""
    from oracle import ref_workloads as RW
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        r = RW.run(rwl, n_samples, sample_offset=i * n_samples, nthreads=nthreads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return n_samples * len(rwl.f) * len(times) / tot, tot / len(times), r


def dump_outputs(out_dir, counters):
    """The counters of the last timed step (what qo_mc_run returns for that sample range) as out_dir/<name>.npy in float64, exact
    below 2**53.  The sample ranges depend on the arguments alone, so two builds run with the same arguments must write equal files."""
    os.makedirs(out_dir, exist_ok=True)
    for name in ("n_pass", "n_total", "fail_per_spec", "hist"):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(counters[name], dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        # the sampler also sees idle gaps; "under load" = samples in the upper half of the power range
        load = [s for s, p in zip(sm, pw) if pw and p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, rank, world):
    """The reference arm: the CPU oracle port on ALL host cores of the box, on a bounded sample of the arm's own workload.
    Rank 0 alone runs it; nothing of the product (qo100net, libqo100net.so) is imported on this path."""
    if rank != 0:
        return
    nthr = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(nthr)        # before the oracle (libgomp) is loaded; torchrun had set it to 1
    os.environ.pop("OMP_THREAD_LIMIT", None)
    from oracle import ref_workloads as RW
    rwl = RW.get(args.workload, NF)
    n = REF_SAMPLES_PER_STEP
    v, per_step, last = cpu_reference(rwl, n, args.steps, args.warmup, nthr)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": rwl.name, "nf": NF, "elements": len(rwl.elems), "samples_per_step": n,
                       "bounded_sample": "%d samples per step instead of the workload's 1e6 per GPU (rate metric: evals/s does not "
                                         "depend on the sample count); host cores do not scale with --gpus" % n,
                       "note": "the reference tree holds no evaluator for this path (external GUI tools); this is the CPU oracle "
                               "port of the same models (oracle/qo100ref.c), OpenMP over samples on all host cores, network built "
                               "by the oracle's own synthesis (oracle/ref_workloads.py): the product library is not loaded"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": nthr, "kind": "port",
                             "sample": "%d samples x %d freq per step, %d steps" % (n, NF, args.steps)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def emit(line):
    """the ONE JSON line, on the process's real stdout"""
    REAL_STDOUT.write(json.dumps(line) + "\n")
    REAL_STDOUT.flush()


def north_star_job(Q, qd, torch, ctx, stream, dist, rank, world, barrier, peak, total):
    """BASELINE config 5 as north_star states it: `total` samples x 4096 points, sharded over the ranks (strong scaling), one
    launch per rank + the counter all-reduce; device time, max over ranks."""
    from qo100net import workloads as W
    wl = W.cfg5(total, NF)
    lo, hi = qd.shard_range(total, rank, world)
    plan = Q.Plan(ctx, wl.net, wl.f, wl.specs, seed=wl.seed, tols=wl.tols, **wl.hist)
    cnt = torch.zeros(plan.num_counters, dtype=torch.int64, device="cuda")
    with torch.cuda.stream(stream):
        for i in range(2):                                  # warm-up on a disjoint sample range
            plan.launch(total + i * 200000, 200000, cnt.data_ptr())
        cnt.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(stream)
        plan.launch(lo, hi - lo, cnt.data_ptr())
        qd.allreduce_counters(cnt)
        b.record(stream)
        barrier()
    ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    sec = float(ms.item()) * 1e-3
    c = qd.split_counters(cnt.cpu(), len(wl.specs), wl.hist["hist_bins"])
    kname, tfi = plan.kernel_name, plan.tf_info
    plan.close()
    evals = total * NF
    out = {"workload": wl.name, "samples_total": total, "nf": NF, "n_gpus": world, "scaling": "strong",
           "samples_this_rank": hi - lo, "seconds": sec, "evals_per_s": evals / sec, "kernel": kname,
           "kernel_plan": tfi if kname in TF_KERNELS else None,
           "n_pass": c["n_pass"], "n_total": c["n_total"], "fail_per_spec": c["fail_per_spec"], "hist_mass": int(sum(c["hist"])),
           "yield": c["n_pass"] / max(1, c["n_total"]),
           "target": "north_star: 1e8 x 4096 on 8 x B200 at >= 50 % of aggregate FP64 FMA peak = 0.96 s (ladder, ALG-v1 349 flops/eval) "
                     "... 1.22 s (with the coupler block, 445 flops/eval)",
           "alg_v1_flops_per_eval": 445.0}
    if peak:
        out["alg_v1_ratio"] = 445.0 * evals / sec * 1e-12 / (peak * world)
        out["executed"] = executed_view(kname, wl.name, evals / sec / world, peak)
    return out


def single_process_ctx_leg(Q, ngpus, n_samples, expect=None):
    """The in-library multi-GPU path (qo_ctx_create(N): one process, samples sharded over N devices, ncclAllReduce of the u64
    counters) on config 5; returns its counters and seconds."""
    from qo100net import workloads as W
    wl = W.cfg5(n_samples, NF)
    ctx = Q.Context(ngpus=ngpus)
    try:
        ctx.mc_run(wl.net, wl.f, wl.specs, wl.seed, 65536, wl.tols, sample_offset=n_samples, **wl.hist)      # warm-up
        t0 = time.perf_counter()
        r = ctx.mc_run(wl.net, wl.f, wl.specs, wl.seed, n_samples, wl.tols, **wl.hist)
        dt = time.perf_counter() - t0
    finally:
        ctx.close()
    out = {"api": "qo_ctx_create(%d) + qo_mc_run: one process, ncclCommInitAll + ncclAllReduce(u64 counters)" % ngpus,
           "workload": wl.name, "samples": n_samples, "n_pass": int(r["n_pass"]), "n_total": int(r["n_total"]),
           "fail_per_spec": [int(x) for x in r["fail_per_spec"]], "wall_seconds": dt, "evals_per_s": n_samples * NF / dt}
    if expect is not None:
        out["equals_sharded_run"] = bool(out["n_pass"] == expect["n_pass"] and out["n_total"] == expect["n_total"] and
                                         out["fail_per_spec"] == [int(x) for x in expect["fail_per_spec"]])
    return out


def nodal_leg(Q, ctx):
    """Row N4 (SURVEY 8f): Monte-Carlo yield of the reference's 5-port bias network (util/pa-bias-simulation/pa-bias-simulation.sch:
    19-72, 23 unknowns, every R +-1 % and C +-5 %) on |S21| and |S31|, 500 000 samples x 1000 points -- the size at which the
    library compiles the job's factorisation plan into a kernel of its own (NVRTC) -- next to the interpreted static-plan kernel."""
    import numpy as np
    from qo100net import workloads as W
    g = np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))        # the measured inductor of pa-bias-simulation.sch:39
    nd, _br, tols = W.pa_bias_nodal(Q, g["11SQ39N_f"], g["11SQ39N_s"])
    nf, n = 1000, 500000
    f = Q.grid_lin(1e8, 3e9, nf)
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, -3.0), (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, -25.0)]
    hist = dict(hist_bins=64, hist_spec=0, hist_lo=-6.0, hist_hi=0.0)
    out = {"workload": "pa-bias 5-port network, 23 unknowns, %d samples x %d points, yield on S21 and S31" % (n, nf), "unit": "points/s"}
    saved = os.environ.pop("QO100NET_NODAL", None)
    try:
        compile_s, best = 0.0, None
        for rep in range(3):
            r = ctx.nodal_mc_run(nd, f, specs, 5, n, tols, sample_offset=rep * n, **hist)
            compile_s = max(compile_s, ctx.nodal_last_compile_seconds())
            best = r if best is None or r["seconds"] < best["seconds"] else best
        out.update({"kernel": ctx.nodal_last_kernel(), "value": n * nf / best["seconds"], "kernel_seconds": best["seconds"],
                    "compile_seconds_first_call": compile_s, "n_pass": int(best["n_pass"]), "n_total": int(best["n_total"])})
        os.environ["QO100NET_NODAL"] = "static"
        ni = 100000
        ctx.nodal_mc_run(nd, f, specs, 5, 512, tols, **hist)
        ri = ctx.nodal_mc_run(nd, f, specs, 5, ni, tols, **hist)
        out["interpreted_plan"] = {"kernel": ctx.nodal_last_kernel(), "value": ni * nf / ri["seconds"]}
    finally:
        os.environ.pop("QO100NET_NODAL", None)
        if saved is not None:
            os.environ["QO100NET_NODAL"] = saved
        nd.close()
    return out


def chain_jit_leg(Q, torch, ctx, stream):
    """What the polynomial kernels cannot take (a line inside the ladder with a measured two-port behind it,
    util/pa-bias-simulation/pa-bias-simulation.sch:39; configs 2 and 5 kept off them; config 5 written out in full): the run-time
    compiled chain kernel (qo_chain_jit.h) next to the opcode interpreter, counters compared (tools/chain_jit_speed.py)."""
    from tools.chain_jit_speed import measure
    saved = {k: os.environ.pop(k, None) for k in ("QO100NET_CHAIN", "QO100NET_KERNEL")}
    try:
        rows = measure(Q, torch, ctx, stream, samples=100000, fs_samples=8192)
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v
    out = {"unit": "evals/s", "jobs": []}
    for name, r in rows.items():
        j = {"job": name, "kernel": r["jit"]["kernel"], "value": r["jit"]["evals_per_s"], "interpreter": r["interp"]["evals_per_s"],
             "speedup": r["speedup"]}
        if "counters_equal" in r:
            j["counters_equal_interpreter"] = r["counters_equal"]
            j["compile_seconds_first_launch"] = r["jit"]["first_launch_s"]
        else:
            j["gb_per_s"] = r["jit"]["gb_per_s"]
            j["max_abs_diff_vs_interpreter"] = r["max_abs_diff"]
        out["jobs"].append(j)
    return out


def full_s_leg(Q, torch, ctx, stream):
    """HBM-bound mode (BASELINE config 4): the full S-matrix written out, 64 B/eval, at the named shape -- 65 536 samples x 4096
    points per filter (17.2 GB), all four filters of the GPSDO bank."""
    from qo100net import workloads as W
    ns = 65536
    buf = torch.empty((4, ns, NF, 2), dtype=torch.float64, device="cuda")
    per, tot_ms = [], 0.0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for w4 in W.cfg4(ns, NF):
        p4 = Q.Plan(ctx, w4.net, w4.f, [], seed=w4.seed, tols=w4.tols, mode=Q.MODE_FULL_S)
        with torch.cuda.stream(stream):
            for _ in range(2):
                p4.launch(0, ns, None, buf.data_ptr())
            torch.cuda.synchronize()
            a.record(stream)
            for _ in range(3):
                p4.launch(0, ns, None, buf.data_ptr())
            b.record(stream)
            torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 3
        tot_ms += ms
        per.append({"workload": w4.name, "kernel": p4.kernel_name, "ms": ms, "gbs": ns * NF * 64 / (ms * 1e-3) * 1e-9})
        p4.close()
    # what a pure write stream reaches on this GPU, same buffer (the copy figure of MEASURED_PEAKS.json is half reads)
    with torch.cuda.stream(stream):
        buf.zero_()
        torch.cuda.synchronize()
        a.record(stream)
        for _ in range(3):
            buf.zero_()
        b.record(stream)
        torch.cuda.synchronize()
    fill_gbs = buf.numel() * 8 / (a.elapsed_time(b) / 3 * 1e-3) * 1e-9
    del buf
    hbm = None
    try:
        hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    gbs = len(per) * ns * NF * 64 / (tot_ms * 1e-3) * 1e-9
    return {"bound": "hbm", "workload": "cfg4 GPSDO bank, FULL_S: 4 filters x 65536 samples x 4096 points, 17.2 GB written per launch (> L2)",
            "achieved": gbs, "peak": hbm or 6650.0, "unit": "GB/s", "frac": gbs / (hbm or 6650.0),
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if hbm else "fallback 6.65 TB/s (B200_PROFILING.md)",
            "evals_per_s": len(per) * ns * NF / (tot_ms * 1e-3), "traffic": None, "per_filter": per,
            "write_only_fill_gbs": fill_gbs, "frac_of_write_only_fill": gbs / fill_gbs,
            "note": "peak is the COPY bandwidth of MEASURED_PEAKS.json (half reads, half writes); this mode only writes, and a plain "
                    "fill of the same buffer (write_only_fill_gbs, measured here) is the tighter roof"}


def main():
    # native libraries write banners to fd 1 (NCCL: "NCCL version ..."): keep the real stdout for the JSON line only and
    # send everything else to stderr
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg5"])
    ap.add_argument("--samples", type=int, default=SAMPLES_PER_GPU, help="samples per GPU per step")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip the north-star job, chain-kernel, CPU and FULL_S legs")
    ap.add_argument("--north-star-samples", type=int, default=NORTH_STAR_SAMPLES)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the counters of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else max(args.warmup, 1)

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import qo100net as Q
    from qo100net import dist as qd
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libqo100net has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        dist = qd.init_process_group("nccl")

    nspg = args.samples
    wl = workload(args.workload, nspg)
    nf = len(wl.f)
    ctx = Q.Context(device=local)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    plan = Q.Plan(ctx, wl.net, wl.f, wl.specs, seed=wl.seed, tols=wl.tols, **wl.hist)
    ncnt = plan.num_counters
    counters = torch.zeros(ncnt, dtype=torch.int64, device="cuda")
    evals_per_step = nspg * nf * world

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i):
        """one pass: this rank's 1e6 samples of global step i, then the counter all-reduce"""
        counters.zero_()
        off = (i * world + rank) * nspg
        plan.launch(off, nspg, counters.data_ptr())
        qd.allreduce_counters(counters)

    sampler = ClockSampler(local) if rank == 0 else None
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            step(i)
        barrier()
        if sampler:
            sampler.start()
        launches0 = plan.launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        ev0.record(stream)
        for i in range(args.steps):
            counters.zero_()
            off = ((args.warmup + i) * world + rank) * nspg
            kev[i][0].record(stream)
            plan.launch(off, nspg, counters.data_ptr())
            kev[i][1].record(stream)
            qd.allreduce_counters(counters)
        ev1.record(stream)
        barrier()
        ms_total = ev0.elapsed_time(ev1)
        kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
        launches = plan.launches - launches0
        last = qd.split_counters(counters.cpu(), len(wl.specs), wl.hist["hist_bins"])
        # end to end through the host-buffer C-ABI call (qo_mc_run): per step H2D of the tables / specs / program, kernel,
        # D2H of the counters; N > 1 adds the all-reduce of the host result
        h2d = plan.h2d_bytes                     # what qo_mc_run copies per call: frequency tables, spec masks, device program
        d2h = ncnt * 8
        for i in range(2):
            ctx.mc_run(wl.net, wl.f, wl.specs, wl.seed, nspg, wl.tols, sample_offset=rank * nspg, **wl.hist)
        # N > 1: the host results are summed across ranks through one reused pinned buffer (H2D, all-reduce, D2H per step)
        hc_pin = torch.zeros(2 + len(wl.specs) + wl.hist["hist_bins"], dtype=torch.int64).pin_memory() if dist is not None else None
        hc_dev = torch.zeros_like(hc_pin, device="cuda") if dist is not None else None
        hc_np = hc_pin.numpy() if dist is not None else None
        ns_ = len(wl.specs)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            r = ctx.mc_run(wl.net, wl.f, wl.specs, wl.seed, nspg, wl.tols, sample_offset=((100 + i) * world + rank) * nspg, **wl.hist)
            if dist is not None:
                hc_np[0], hc_np[1] = r["n_pass"], r["n_total"]
                hc_np[2:2 + ns_] = r["fail_per_spec"]
                hc_np[2 + ns_:] = r["hist"]
                hc_dev.copy_(hc_pin, non_blocking=True)
                qd.allreduce_counters(hc_dev)
                hc_pin.copy_(hc_dev, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        barrier()
        e2e_s = time.perf_counter() - t0
        clocks = sampler.stop() if sampler else None       # sampled over both timed regions (resident steps and end-to-end steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)

    tm = torch.tensor([ms_total, e2e_s * 1e3, kernel_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, kernel_ms = [float(x) for x in tm.cpu()]
    value = evals_per_step * args.steps / (ms_total * 1e-3)
    e2e_value = evals_per_step * args.steps / (e2e_ms * 1e-3)

    peak = ctx.measure_dfma_peak()                      # TFLOP/s, measured now on this rank's GPU
    ns_job = None
    if not args.no_extras:
        try:
            ns_job = north_star_job(Q, qd, torch, ctx, stream, dist, rank, world, barrier, peak, args.north_star_samples)
        except Exception as ex:                         # a secondary leg must never take the headline line down
            ns_job = {"error": str(ex)}

    # the in-library multi-GPU path: rank 0 alone drives all N GPUs from one process while the other ranks wait on the store
    ctx_leg = None
    if not args.no_extras and world > 1:
        store = None
        try:
            from torch.distributed import distributed_c10d as c10d
            store = c10d._get_default_store()
        except Exception:
            store = None
        if store is not None:
            if rank == 0:
                try:
                    n_ctx = 8000000
                    from qo100net import workloads as W
                    w5 = W.cfg5(n_ctx, NF)
                    ref = ctx.mc_run(w5.net, w5.f, w5.specs, w5.seed, n_ctx, w5.tols, **w5.hist)      # the same range on ONE device
                    ctx_leg = single_process_ctx_leg(Q, world, n_ctx, expect=ref)
                except Exception as ex:
                    ctx_leg = {"error": str(ex)}
                store.set("qo_ctx_leg_done", "1")
            else:
                store.wait(["qo_ctx_leg_done"])

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    flops = plan.flops_per_eval
    evals_per_launch = nspg * nf
    rate_gpu = evals_per_launch / (kernel_ms * 1e-3)
    alg_tflops = flops * rate_gpu * 1e-12
    ex = executed_view(plan.kernel_name, wl.name, rate_gpu, peak)
    prof = executed_profile(plan.kernel_name, wl.name) or {}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.name, "samples_per_gpu_per_step": nspg, "nf": nf, "elements": len(wl.net),
                   "flops_per_eval_alg_v1": flops, "parallelism": "samples sharded x%d, u64 counter all-reduce" % world,
                   "l2": "no flush: the reduce-only path reads < 200 KB of tables by design (bytes/eval ~ 0); every "
                         "step draws a fresh global sample range",
                   "kernel_plan": plan.tf_info if plan.kernel_name in TF_KERNELS else None,
                   "yield_last_step": last["n_pass"] / max(1, last["n_total"])},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "qo_mc_run (host buffers)"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "fp64_fma", "achieved": ex["tflops"] if ex else None, "peak": peak, "unit": "TFLOP/s",
                     "frac": ex["frac_of_peak"] if ex else None,
                     "traffic": prof.get("dram_bytes_per_launch"), "kernel": plan.kernel_name, "kernel_ms": kernel_ms,
                     "executed": ex,
                     "alg_v1_tflops": alg_tflops, "alg_v1_ratio": alg_tflops / peak,
                     "note": "achieved = EXECUTED FP64 flops per eval (ncu smsp__sass_thread_inst_executed_op_{dfma,dmul,dadd}_pred_on "
                             "of this kernel on this workload, DFMA = 2: profiles/executed_fp64.json) x evals / kernel time measured "
                             "here (a step launches the thread-per-sample kernel for all whole 32-sample batches and the warp-per-"
                             "sample kernel for the few samples left; kernel_ms covers both); frac = achieved / peak.  alg_v1_ratio = SURVEY 8d's algorithmic count (a 2x2 complex chain step "
                             "and a complex divide per element, 349 flops/eval) at the same rate over the same peak: above 1 because "
                             "the transfer-function kernel expands the cascade into real polynomials once per sample and runs Horner "
                             "per point, i.e. it does less work than ALG-v1 counts.  chain_kernel = the same job on the straight-line "
                             "ABCD-chain kernel (QO100NET_KERNEL=ladder), whose executed work is close to ALG-v1.",
                     "peak_source": "measured in this run: qo_measure_dfma_peak (8 independent DFMA chains/thread, "
                                    "best of 5); MEASURED_PEAKS.json has no FP64 figure (nominal 37.2 TFLOP/s)"},
    }
    if ns_job is not None:
        line["north_star_job"] = ns_job
    if ctx_leg is not None:
        line["single_process_ctx"] = ctx_leg
    if not args.no_extras and plan.kernel_name in TF_KERNELS:
        # the same workload on the other kernels, for comparison: warp-per-sample polynomial kernel (round 1's headline kernel)
        # and the straight-line ABCD-chain kernel (north_star (c) as worded)
        for key, force in (("warp_per_sample_kernel", "tf"), ("chain_kernel", "ladder")):
            os.environ["QO100NET_KERNEL"] = force
            try:
                p2 = Q.Plan(ctx, wl.net, wl.f, wl.specs, seed=wl.seed, tols=wl.tols, **wl.hist)
                c2 = torch.zeros(ncnt, dtype=torch.int64, device="cuda")
                ms2 = time_plan(p2, stream, c2, nspg, max(3, args.steps // 2), 2, torch)
                r2 = evals_per_launch / (ms2 * 1e-3)
                line["roofline"][key] = {"kernel": p2.kernel_name, "kernel_ms": ms2, "evals_per_s_per_gpu": r2,
                                         "alg_v1_tflops": flops * r2 * 1e-12, "alg_v1_ratio": flops * r2 * 1e-12 / peak,
                                         "executed": executed_view(p2.kernel_name, wl.name, r2, peak)}
                p2.close()
            except Exception as ex2:
                line["roofline"][key] = {"error": str(ex2)}
            finally:
                os.environ.pop("QO100NET_KERNEL", None)
    if not args.no_extras and world == 1:
        # CPU baseline on a bounded sample of the same workload (rank 0, N = 1 only), oracle-built network
        try:
            from oracle import ref_workloads as RW
            nthr = host_cores()
            rwl = RW.get(args.workload, NF)
            n = 40000
            v, _, _ = cpu_reference(rwl, n, 2, 1, nthr)
            v1, _, _ = cpu_reference(rwl, 2000, 1, 0, 1)          # the "single-threaded C loop over the same model" of north_star
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": nthr, "kind": "port",
                                    "sample": "%d samples x %d freq, 2 timed passes, OpenMP over samples" % (n, nf),
                                    "single_thread": {"value": v1, "unit": UNIT, "cores": 1, "sample": "2000 samples x %d freq, 1 pass" % nf}}
        except Exception as ex3:
            line["cpu_baseline"] = {"error": str(ex3)}
        try:
            line["roofline_hbm"] = full_s_leg(Q, torch, ctx, stream)
        except Exception as ex4:
            line["roofline_hbm"] = {"error": str(ex4)}
        try:
            line["nodal"] = nodal_leg(Q, ctx)
        except Exception as ex5:
            line["nodal"] = {"error": str(ex5)}
        try:
            line["chain_jit"] = chain_jit_leg(Q, torch, ctx, stream)
        except Exception as ex6:
            line["chain_jit"] = {"error": str(ex6)}
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
