#!/usr/bin/env python
"""bench.py — throughput of the lineage-forest log-likelihood (FP64) on N B200s.

Workload (BASELINE.json configs[1]): synthetic forest of 10 000 lineage trees x 6 generations x ~20 points
per cell PER GPU (630 000 cells, ~12.6 M cell-timepoints), one log-likelihood evaluation per step,
"gauss" division, "const" noise, fresh mode.  Weak scaling: every rank simulates its own forest (seed + rank);
the init_cells_f/r population statistics are combined across ranks (all-reduce of 10 sums) and the scalar
log-likelihood is all-reduced every step (NCCL).  Inputs (353 MB/GPU) are larger than the 126 MB L2.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (CUDA kernels through the C ABI)
  python bench.py --impl reference ...                         the reference's CPU math on the host cores
  python bench.py ... --dump-outputs DIR                       also write the last timed step's log-likelihoods to DIR/*.npy

One JSON line on stdout (rank 0).
  value / ms_per_step   cell-timepoints/s of the whole job with the forest resident in HBM, in the library's FAST likelihood
                        mode (quadrature + FMA; its gate |dloglik| / |loglik| <= 1e-10 against the reference is evaluated in
                        this run, `parity`, and the headline falls back to the strict mode if it is not met)
  strict                the same with the STRICT kernels (bit-identical to the reference's arithmetic)
  e2e                   through the host-buffer C-ABI call: this step's measurements (log_length, fp; the time grid of an
                        unchanged genealogy does not travel again) uploaded from pinned host memory + ggp_loglik (host
                        parameters in, host result out), wall clock
  e2e_resident          ggp_loglik(host parameters -> host result) on the resident forest: what -m / -s do per evaluation
  roofline              FP64-pipe fraction of the headline kernel (F_alg = 3 700 flop per cell-timepoint, SURVEY.md 8d, against
                        the DFMA peak measured in this process); roofline_strict the same for the strict kernel
  parity                GPU (strict and fast) against the CPU baseline's own result on the SAME trees
  cpu_baseline          the reference's math on one host core (warm-up + median of 5)
  configs               BASELINE configs[2..4] on this GPU (short runs): -p on a 1 M-cell forest, a 256-vector slice of the
                        4096-vector scan, -j on a 100 k-cell forest with two segments; and configs[0], the reference's example data
                        set (evaluation latency, the command line's -m -p in the fast mode)
  strong                (N > 1) ONE 10 000-tree forest partitioned over the ranks: strong scaling of the same evaluation
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_ALG = 3700.0        # algorithmic FP64 flop per cell-timepoint per directional pass (SURVEY.md 8d, DESIGN.md)
F_ALG_PREDICT = 8900.0   # -p: 2 F_alg + 1 500 (combine)
F_ALG_JOINT = 5500.0     # -j: per emitted joint
B_ALG = 28.0          # algorithmic bytes per cell-timepoint: time, x, g (f64) + segment (i32)
# dram__bytes_read.sum + dram__bytes_write.sum per cell-timepoint from the ncu --set full captures of the largest
# generation's launch (6 399 691 ctp): strict profiles/r01_s5_loglik_coop_gen5.txt, fast profiles/r02_fast5_final_gen5.txt
DRAM_BYTES_PER_CTP_NCU = {"strict": (204.285440e6 + 4.971776e6) / 6399691.0, "fast": (130.749952e6 + 4.492032e6) / 6399691.0}
# what the fast kernel EXECUTES per cell-timepoint with the 5-node rule (same capture: 59.53 M DFMA, 21.71 M DMUL, 9.77 M DADD
# warp instructions for 6 399 691 ctp), an FMA counted as two flops
FAST_EXEC = {"nodes": 5, "dfma": 59528912 * 32 / 6399691.0, "dmul": 21709416 * 32 / 6399691.0, "dadd": 9770336 * 32 / 6399691.0,
             "instr": 129461032 * 32 / 6399691.0, "fp64_pipe_busy": 0.704}
METRIC = "cell-timepoints/s, FP64 log-likelihood evaluation (loglik evals/s in config)"
GATE = 1e-10          # north star: log-likelihood within relative 1e-10 of the reference


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--trees", type=int, default=10000)
    ap.add_argument("--generations", type=int, default=6)
    ap.add_argument("--cpu-sample-trees", type=int, default=600)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2..4] extras")
    ap.add_argument("--mode", default="auto", choices=["auto", "fast", "strict"], help="headline kernel (auto: fast if its gate is met)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the log-likelihood the last timed step returned as DIR/loglik_<mode>.npy "
                         "(float64, one per timed mode), so that two builds can be compared on the same seeded inputs")
    return ap.parse_args()


def dump_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, value in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(value, dtype=np.float64))


def workload_config(args, world, extra=None):
    c = {"workload": "configs[1]: synthetic forest %d trees x %d generations x ~20 pts/cell per GPU, single "
                     "log-likelihood eval, gauss division, const noise, fresh mode" % (args.trees, args.generations),
         "trees_per_gpu": args.trees, "generations": args.generations, "n_vec": 1, "parallelism": "trees sharded x%d" % world,
         "l2": "inputs (28 B/ctp, ~353 MB per GPU) larger than the 126 MB L2"}
    if extra:
        c.update(extra)
    return c


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's filter loop around the reference's own mean_cov_model.h +
# Faddeeva.cc (oracle/_ref) where that build exists, else the oracle port
# ---------------------------------------------------------------------------------------------------
def _cpu_worker(q_in, q_out, use_ref):
    from oracle import oracle_py
    if use_ref:
        oracle_py.use_reference_math(True)
    import gfp_gaussian_process_b200 as ggp
    o = None
    while True:
        msg = q_in.get()
        if msg is None:
            break
        if msg[0] == "load":
            z = np.load(msg[1])
            data = ggp.LineageData(cell_offset=z["cell_offset"], parent=z["parent"], time=z["time"], log_length=z["log_length"],
                                   fp=z["fp"], noise_model="const", division_model="gauss", init_f=z["init_f"], init_r=z["init_r"])
            o = oracle_py.Oracle(data)
            q_out.put(("loaded", data.n_ctp))
        else:
            t = time.perf_counter()
            ll = o.total_loglik(msg[1])
            q_out.put((ll, time.perf_counter() - t))


def cpu_pool_bench(data, params, n_proc, trees_per_proc, steps, warmup, use_ref):
    """P processes, each evaluating its own shard of `trees_per_proc` trees per step; returns (ctp/s, ctp per step, loglik)"""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    roots = data.roots()
    init_f, init_r = data.init_stats()
    procs, files, total = [], [], 0
    tmp = tempfile.mkdtemp(prefix="ggp_bench_")
    for r in range(n_proc):
        sub, _, _ = data.subset(roots[r * trees_per_proc:(r + 1) * trees_per_proc])
        fn = os.path.join(tmp, f"shard{r}.npz")
        np.savez(fn, cell_offset=sub.cell_offset, parent=sub.parent, time=sub.time, log_length=sub.log_length, fp=sub.fp,
                 init_f=init_f, init_r=init_r)
        files.append(fn)
        qi, qo = ctx.Queue(), ctx.Queue()
        p = ctx.Process(target=_cpu_worker, args=(qi, qo, use_ref), daemon=True)
        p.start()
        procs.append((p, qi, qo))
    for (p, qi, qo), fn in zip(procs, files):
        qi.put(("load", fn))
    for p, qi, qo in procs:
        total += qo.get()[1]
    times, ll = [], 0.0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for p, qi, qo in procs:
            qi.put(("eval", params))
        res = [qo.get() for p, qi, qo in procs]
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        ll = sum(r[0] for r in res)
    for p, qi, qo in procs:
        qi.put(None)
    for p, qi, qo in procs:
        p.join(timeout=10)
    for fn in files:
        os.remove(fn)
    os.rmdir(tmp)
    return total * len(times) / sum(times), total, ll, sum(times) / len(times)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import gfp_gaussian_process_b200 as ggp
    from oracle import oracle_py
    use_ref = oracle_py.use_reference_math(True)
    oracle_py.use_reference_math(False)
    cores = min(host_cores(), 64)
    trees_per_proc = 120          # ~150 k ctp, ~0.5 s per process per step
    data = ggp.simulate_forest(cores * trees_per_proc, args.generations, seed=20261018)
    steps, warmup = args.steps, args.warmup   # the same counts as the GPU arm; a step is a bounded sample
    v, ctp, ll, t = cpu_pool_bench(data, ggp.PARAMS_CONST_GAUSS, cores, trees_per_proc, steps, warmup, use_ref)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"loglik_reference": [ll]})
    kind = "reference" if use_ref else "port"
    sample = ("%d trees x %d generations (%d ctp) of the configs[1] forest per step, %d processes x %d trees; %s"
              % (cores * trees_per_proc, args.generations, ctp, cores, trees_per_proc,
                 "reference mean_cov_model.h + Faddeeva.cc compiled unmodified (oracle/_ref) inside the oracle's filter loop, which "
                 "equals the reference's own likelihood.h / predictions.h bit for bit (tests/test_ref_wrappers.py)" if use_ref
                 else "oracle port (oracle/ggp_oracle.cpp)"))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "ctp/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(args, world, {"reference_sample_trees_per_process": trees_per_proc, "reference_processes": cores,
                                                    "reference_sample_ctp_per_step": int(ctp)}),
            "cpu_baseline": {"value": v, "unit": "ctp/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "ctp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "loglik_evals_per_s_full_forest": v / (args.trees * (2 ** args.generations - 1) * 20.0), "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.p = None
        self.f = None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, power, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "power_w_max": float(max(power)), "samples": len(sm)}
        return out


def global_init_stats(data, world, torch, dist):
    """population statistics over ALL ranks' cells (moma_input.h:675-735): all-reduce of counts and sums"""
    n = np.diff(data.cell_offset)
    sel = n > 1
    sums = []
    for idx in (data.cell_offset[:-1][sel], data.cell_offset[1:][sel] - 1):
        x, g = data.log_length[idx], data.fp[idx]
        sums += [float(len(idx)), x.sum(), g.sum(), (x * x).sum(), (g * g).sum()]
    st = torch.tensor(sums, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(st)
    st = st.cpu().numpy()
    out = []
    for k in (0, 5):
        c, sx, sg, sxx, sgg = st[k:k + 5]
        out.append(np.array([sx / c, sg / c, sxx / c - (sx / c) ** 2, sgg / c - (sg / c) ** 2]))
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import gfp_gaussian_process_b200 as ggp
    from gfp_gaussian_process_b200 import _lib, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this implementation has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # stdout carries exactly one JSON line: native libraries that print there (NCCL's version banner) go to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    P = ggp.PARAMS_CONST_GAUSS
    dp = _lib.c_double_p

    data = ggp.simulate_forest(args.trees, args.generations, seed=20261018 + rank)
    data.init_f, data.init_r = global_init_stats(data, world, torch, dist)
    forest = ggp.Forest(data, device=local)
    stream = torch.cuda.current_stream()
    forest.set_stream(stream.cuda_stream)
    n_ctp = forest.n_ctp
    n_cells_gpu = forest.n_cells
    d_params = torch.tensor(P, dtype=torch.float64, device="cuda").reshape(1, 11)
    d_out = torch.zeros(1, dtype=torch.float64, device="cuda")
    total = torch.zeros(1, dtype=torch.float64, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t)
        return float(t.item())

    ctp_total = allsum(float(n_ctp))

    def timed_resident(fr, steps, warmup, sample_clocks=False):
        """K steps of (device-resident evaluation + all-reduce of the scalar), CUDA events on the stream, max over ranks"""
        def step():
            _lib.check(lib.ggp_loglik_device(fr.handle, d_params.data_ptr(), 1, d_out.data_ptr()))
            total.copy_(d_out)
            if world > 1:
                dist.all_reduce(total)
        for _ in range(warmup):
            step()
        barrier()
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
            time.sleep(0.3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = fr.last_launch_count * steps
        if sampler:
            time.sleep(0.2)
        clocks = sampler.stop() if sampler else None
        k = np.zeros(1)
        _lib.check(lib.ggp_sync_kernel_ms(fr.handle, k.ctypes.data_as(dp)))   # also checks the fast mode's validity flags
        # kernel-only time (events inside the library, same stream), separate loop so that the event sync is outside the timed region
        kern = []
        for _ in range(steps):
            _lib.check(lib.ggp_loglik_device(fr.handle, d_params.data_ptr(), 1, d_out.data_ptr()))
            _lib.check(lib.ggp_sync_kernel_ms(fr.handle, k.ctypes.data_as(dp)))
            kern.append(float(k[0]))
        return allmax(ms) / steps, float(np.mean(kern)), int(launches), float(total.item()), clocks

    # end to end through the host-buffer C-ABI calls
    pin = [torch.from_numpy(a).pin_memory() for a in (data.log_length, data.fp)]

    def timed_e2e(fr, steps, upload):
        def step():
            if upload:   # this step's measurements; the time grid of the unchanged genealogy stays; statistics travel with the data
                fr.upload_series(None, pin[0].data_ptr(), pin[1].data_ptr(), data.init_f, data.init_r)
            return ggp.total_likelihood(P, fr)
        for _ in range(2):
            ll = step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            ll = step()
        torch.cuda.synchronize()
        return allmax((time.perf_counter() - t0) / steps), allsum(ll)

    # the end-to-end step's roofline: the same two pinned arrays copied to the device with nothing else going on (PCIe alone)
    def timed_pcie_copy(reps):
        dev = [torch.empty(a.shape, dtype=a.dtype, device="cuda") for a in pin]
        ts = []
        for _ in range(reps + 3):
            barrier()   # all ranks copy at the same time: at N > 1 this is the host-side ceiling the end-to-end step shares
            t0 = time.perf_counter()
            for dst, src in zip(dev, pin):
                dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        # the link's capability: the best repetition (a GPU that has idled copies at 43 instead of 55 GB/s for a while)
        return allmax(float(np.min(ts[3:])))

    res = {}
    for mode in ("strict", "fast"):
        forest.set_mode(mode)
        ggp.total_likelihood(P, forest)   # fast: the library picks the quadrature order from these parameters and the forest's dt
        ms_step, kern_ms, launches, ll, clocks = timed_resident(forest, args.steps, args.warmup, sample_clocks=True)
        e2e_s, ll_e2e = timed_e2e(forest, args.steps, True)
        res_s, _ = timed_e2e(forest, args.steps, False)
        res[mode] = dict(ms_step=ms_step, kern_ms=kern_ms, launches=launches, loglik=ll, clocks=clocks, e2e_s=e2e_s, loglik_e2e=ll_e2e,
                         resident_s=res_s, reruns=int(forest.last_strict_reruns), nodes=int(forest.last_fast_nodes))
    pcie_copy_s = timed_pcie_copy(8)   # right behind the timed loops: clocks and link are where the end-to-end steps had them
    if args.dump_outputs and rank == 0:
        # the all-reduced total that ggp_loglik_device's caller held after the last timed step of each mode
        dump_outputs(args.dump_outputs, {"loglik_" + mode: [res[mode]["loglik"]] for mode in res})
    gate_full = abs(res["fast"]["loglik"] - res["strict"]["loglik"]) / abs(res["strict"]["loglik"])

    # strong scaling: ONE forest (the rank-0 seed) partitioned over the ranks by tree, statistics of the whole forest
    strong = None
    whole = None
    if world > 1:
        whole = ggp.simulate_forest(args.trees, args.generations, seed=20261018)
        whole.init_f, whole.init_r = whole.init_stats()
        sub, _, _ = sharding.shard(whole, rank, world)
        fs = ggp.Forest(sub, device=local)
        fs.set_stream(stream.cuda_stream)
        strong = {}
        for mode in ("strict", "fast"):
            fs.set_mode(mode)
            ms_s, kern_s, _, ll_s, _ = timed_resident(fs, args.steps, args.warmup)
            strong[mode] = {"ms_per_step": ms_s, "value": whole.n_ctp / (ms_s * 1e-3), "kernel_ms_max_rank": allmax(kern_s), "loglik": ll_s}
        strong["ctp_total"] = int(whole.n_ctp)
        strong["imbalance_max_over_mean_ctp"] = allmax(float(sub.n_ctp)) / (whole.n_ctp / world)
        strong["what"] = ("one %d-tree forest (seed of rank 0) partitioned over %d ranks by greedy bin packing of trees "
                          "(sharding.partition_roots), scalar all-reduce per step; value = ctp of the whole forest / max-over-ranks time"
                          % (args.trees, world))
        fs.close()

    # one process, N GPUs (ggp_group): the other ranks leave, rank 0 drives every device through ONE handle
    one_process = None
    if world > 1:
        forest.close()
        forest = None
        torch.cuda.empty_cache()
        barrier()
        dist.destroy_process_group()
        if rank != 0:
            return
        time.sleep(1.0)   # let the other ranks release their devices
        one_process = measure_one_process(ggp, torch, world, args, whole, P)

    if rank == 0:
        peak = np.zeros(1)
        _lib.check(lib.ggp_fp64_peak(local, peak.ctypes.data_as(dp)))
        fp64_peak = float(peak[0])
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            hbm_peak, hbm_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"

        def executed(r):
            """executed FP64 work of the fast kernel (ncu instruction counts of the 5-node build; other node counts: none)"""
            if r["nodes"] != FAST_EXEC["nodes"]:
                return None
            flop = 2 * FAST_EXEC["dfma"] + FAST_EXEC["dmul"] + FAST_EXEC["dadd"]
            ach = n_ctp * flop / (r["kern_ms"] * 1e-3) / 1e12
            return {"flop_per_ctp": flop, "fp64_instr_per_ctp": FAST_EXEC["dfma"] + FAST_EXEC["dmul"] + FAST_EXEC["dadd"],
                    "instr_per_ctp": FAST_EXEC["instr"], "achieved": ach, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                    "fp64_pipe_busy_ncu": FAST_EXEC["fp64_pipe_busy"]}

        def roofline(mode):
            r = res[mode]
            ach = n_ctp * F_ALG / (r["kern_ms"] * 1e-3) / 1e12
            kernel = (("ggp_fast_loglik_kernel<%d, 3, true> (one thread per cell, %d-node rule; " % (r["nodes"], r["nodes"])) + "%d launches per step)"
                      if mode == "fast" else "ggp_loglik_coop_kernel (four warps per 32 cells; %d launches per step)") % (r["launches"] // args.steps)
            return {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                    "traffic": DRAM_BYTES_PER_CTP_NCU[mode] * n_ctp,
                    "traffic_unit": "bytes per step (ncu dram bytes per ctp of the largest launch x ctp per step)",
                    "kernel": kernel, "kernel_ms_per_step": r["kern_ms"], "flop_per_ctp": F_ALG,
                    "peak_source": "DFMA micro-benchmark run in this process (ggp_fp64_peak); MEASURED_PEAKS.json holds no FP64 figure",
                    "note": ("F_alg counts the reference's formulas (38 integrals via Dawson, 26 exp, 3 pow per step); the fast kernel "
                             "evaluates the same moments by quadrature with 3 N short exponentials and no Dawson / pow, so `frac` is "
                             "ALGORITHMIC work per second over the DFMA peak and exceeds 1; `executed` is what the kernel really does "
                             "(ncu, 5 nodes: 647 instructions / 455 FP64 per ctp, FP64 pipe 70.4 % busy, profiles/r02_fast5_final_gen5.txt)")
                    if mode == "fast" else
                            ("strict arithmetic cannot fuse (FMA off) and evaluates 66 exp + 14 Dawson + 3 pow per step bit for bit: "
                             "3 220 executed FP64 instructions per ctp, FP64 pipe busy 44.5 % (profiles/r01_s5_loglik_coop_gen5.txt)"),
                    "hbm": {"achieved": n_ctp * B_ALG / (r["kern_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": n_ctp * B_ALG / (r["kern_ms"] * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src},
                    **({"executed": executed(r)} if mode == "fast" else {})}

        def e2e(mode):
            r = res[mode]
            return {"value": ctp_total / r["e2e_s"], "unit": "ctp/s", "h2d_bytes_per_step": int(2 * 8 * n_ctp + 88 + 64),
                    "d2h_bytes_per_step": 16, "ms_per_step": r["e2e_s"] * 1e3,
                    "h2d_gbps_per_gpu": 2 * 8 * n_ctp / r["e2e_s"] / 1e9,
                    "pcie": {"copy_alone_ms": pcie_copy_s * 1e3, "copy_alone_gbps_per_gpu": 2 * 8 * n_ctp / pcie_copy_s / 1e9,
                             "frac": pcie_copy_s / r["e2e_s"],
                             "what": "the step's two pinned arrays copied to the device with no kernel running, ALL ranks at the same time "
                                     "(barrier before every copy, max over ranks): the end-to-end step is bound by this path - PCIe at "
                                     "N = 1, the guest's host side at N = 8 (tools/r02_jobs/h2d_concurrent.py: 55 GB/s per GPU alone, "
                                     "23.5 - 36 GB/s with eight copying together); frac = copy alone / whole step"},
                    "what": "ggp_forest_upload_series (this step's log_length and fp from pinned host memory with their init_cells "
                            "statistics; the unchanged time grid is not sent again) + ggp_loglik (host params in, host log-likelihood "
                            "and NaN record out), wall clock around the host calls"}

        line = {"metric": METRIC, "unit": "ctp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "ctp_total": ctp_total, "cells_per_gpu": n_cells_gpu}

        parity = {"gate": GATE, "fast_vs_strict_full_forest": gate_full}
        if not args.no_cpu_baseline and world == 1:
            from oracle import oracle_py
            use_ref = oracle_py.use_reference_math(True)
            sub, cells, _ = data.subset(data.roots()[:args.cpu_sample_trees])
            sub.init_f, sub.init_r = data.init_f, data.init_r
            o = oracle_py.Oracle(sub)
            ts = []
            for it in range(6):   # one warm-up + median of 5
                t0 = time.perf_counter()
                ll_cpu, pc_cpu = o.total_loglik(P, per_cell=True)
                if it:
                    ts.append(time.perf_counter() - t0)
            dt = float(np.median(ts))
            line["cpu_baseline"] = {"value": sub.n_ctp / dt, "unit": "ctp/s", "cores": 1, "kind": "reference" if use_ref else "port",
                                    "sample": "first %d trees (%d ctp) of the same forest, one warm-up + median of 5 evaluations (%.2f s "
                                              "each); %s" % (args.cpu_sample_trees, sub.n_ctp, dt,
                                                             "reference mean_cov_model.h + Faddeeva.cc (oracle/_ref) inside the oracle's filter loop"
                                                             if use_ref else "oracle port"), "loglik": ll_cpu}
            # the GPU on the SAME trees
            fsub = ggp.Forest(sub, device=local)
            ll_g, pc_g = ggp.total_likelihood(P, fsub, per_cell=True)
            fsub.set_mode("fast")
            ll_f = ggp.total_likelihood(P, fsub)
            fsub.close()
            parity.update({"sample": "the cpu_baseline's %d trees" % args.cpu_sample_trees,
                           "rel_err_loglik": abs(ll_g - ll_cpu) / abs(ll_cpu),
                           "cells_bit_equal": int(np.sum(pc_g.view(np.uint64) == pc_cpu.view(np.uint64))), "cells": int(sub.n_cells),
                           "fast_rel_err_loglik": abs(ll_f - ll_cpu) / abs(ll_cpu)})
        gate_ok = gate_full <= GATE and parity.get("fast_rel_err_loglik", 0.0) <= GATE and res["fast"]["reruns"] == 0
        head = "strict" if (args.mode == "strict" or (args.mode == "auto" and not gate_ok)) else "fast"
        parity["fast_gate_met"] = bool(gate_ok)
        r = res[head]
        line.update({
            "value": ctp_total / (r["ms_step"] * 1e-3), "ms_per_step": r["ms_step"],
            "config": workload_config(args, world, {"mode": "%s likelihood kernels (%s)" % (head, ("%d-node quadrature + FMA, gate 1e-10 met in this run" % r["nodes"])
                                                                                             if head == "fast" else "bit-identical to the reference's arithmetic")}),
            "loglik_evals_per_s": 1e3 / r["ms_step"], "loglik": r["loglik"], "loglik_e2e": r["loglik_e2e"], "clocks": r["clocks"],
            "e2e": e2e(head),
            "e2e_resident": {"value": ctp_total / r["resident_s"], "unit": "ctp/s", "ms_per_step": r["resident_s"] * 1e3,
                             "h2d_bytes_per_step": 88, "d2h_bytes_per_step": 16,
                             "what": "ggp_loglik(host params -> host log-likelihood) on the resident forest: one -m / -s evaluation"},
            "gpu_launches": r["launches"], "roofline": roofline(head), "parity": parity})
        other = "strict" if head == "fast" else "fast"
        o_ = res[other]
        line[other] = {"value": ctp_total / (o_["ms_step"] * 1e-3), "ms_per_step": o_["ms_step"], "loglik": o_["loglik"],
                       "e2e": e2e(other), "e2e_resident_ms": o_["resident_s"] * 1e3, "gpu_launches": o_["launches"], "clocks": o_["clocks"]}
        line["roofline_" + other] = roofline(other)
        if strong:
            line["strong"] = strong
        if one_process:
            line["one_process"] = one_process
        if not args.no_configs and world == 1:
            forest.close()
            forest = None
            torch.cuda.empty_cache()
            line["configs"] = measure_configs(ggp, _lib, lib, torch, local, fp64_peak)
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if forest is not None:
        forest.close()


def measure_one_process(ggp, torch, n_dev, args, whole, P):
    """ONE host process driving all N GPUs through the library's group handle (ggp_group): strong scaling of the configs[1]
    evaluation, and configs[2] (-p on 1 M cells) sharded over the devices with every prediction row landing in one pinned
    host buffer (host parameters in, all rows out, wall clock)"""
    out = {"what": "rank 0 alone, ggp_group over %d devices: trees split into contiguous runs, one host thread per shard, log-likelihoods "
                   "added on the host in shard order, prediction rows copied by each device straight into their place" % n_dev}
    g = ggp.ForestGroup(whole, list(range(n_dev)))
    for mode in ("strict", "fast"):
        g.set_mode(mode)
        for _ in range(3):
            ll = g.total_likelihood(P)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ll = g.total_likelihood(P)
        dt = (time.perf_counter() - t0) / args.steps
        out["loglik_" + mode] = {"ms_per_eval": dt * 1e3, "ctp_per_s": whole.n_ctp / dt, "loglik": float(ll)}
    g.close()
    data = ggp.simulate_forest(15873, 6, noise_model="scaled", division_model="binomial", seed=20261018)
    g = ggp.ForestGroup(data, list(range(n_dev)))
    pins = {k: torch.empty((data.n_ctp, 14), dtype=torch.float64).pin_memory().numpy() for k in ("forward", "backward", "prediction")}
    Pp = np.ascontiguousarray(ggp.PARAMS_SCALED_BINOMIAL.reshape(1, 11))
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        g.predictions(Pp, packed=True, out=pins)
        ts.append(time.perf_counter() - t0)
    out["cfg3_predict_sharded"] = {"n_cells": int(data.n_cells), "n_ctp": int(data.n_ctp), "e2e_ms": float(np.min(ts[1:])) * 1e3,
                                   "ctp_per_s": data.n_ctp / float(np.min(ts[1:])), "d2h_bytes": int(3 * 14 * 8 * data.n_ctp),
                                   "finite": bool(np.isfinite(pins["prediction"][::997]).all())}
    g.close()
    # configs[4] (-j on 100 k cells, two segments) with the correlation reduction, every device on its own trees
    P2 = np.stack([ggp.PARAMS_SCALED_BINOMIAL, ggp.PARAMS_SCALED_BINOMIAL * np.array([1, 1, 1, 2, 1, 1, 1, 1, 1, 1, 1.])])
    data = ggp.simulate_forest(1587, 6, params=ggp.PARAMS_SCALED_BINOMIAL, noise_model="scaled", division_model="binomial",
                               seed=20261018, n_segments=2)
    g = ggp.ForestGroup(data, list(range(n_dev)))
    g.predictions(P2, packed=True)
    ts, nj = [], 0
    for _ in range(3):
        t0 = time.perf_counter()
        sums, nj = g.correlation_sums(P2, 15.0, 200)
        ts.append(time.perf_counter() - t0)
    out["cfg5_correlation_sharded"] = {"n_cells": int(data.n_cells), "joints": int(nj), "e2e_ms": float(np.min(ts[1:])) * 1e3,
                                       "joints_per_s": nj / float(np.min(ts[1:])),
                                       "what": "ggp_group_correlation_sums: walk + lag-binned reduction on every device, sums added on the host"}
    g.close()
    return out


def measure_configs(ggp, _lib, lib, torch, device, fp64_peak):
    """BASELINE configs[2..4] on this GPU, short runs (tools/measure_configs.py holds the long forms)"""
    import ctypes as C
    dp = _lib.c_double_p
    out = {}
    # configs[2]: -p on a 1 M-cell forest (one GPU's view; 8 GPUs shard the trees), scaled noise + binomial division
    data = ggp.simulate_forest(15873, 6, noise_model="scaled", division_model="binomial", seed=20261018)
    f = ggp.Forest(data, device=device)
    P = np.ascontiguousarray(ggp.PARAMS_SCALED_BINOMIAL.reshape(1, 11))
    ms = []
    for _ in range(4):
        _lib.check(lib.ggp_predict(f.handle, P.ctypes.data_as(dp), 1, None, None, None))
        ms.append(f.last_kernel_ms)
    kms = float(np.median(ms[1:]))
    pins = {k: torch.empty((data.n_ctp, 14), dtype=torch.float64).pin_memory().numpy() for k in ("forward", "backward", "prediction")}
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        ggp.prediction_upper14(f, P, out=pins)
        ts.append(time.perf_counter() - t0)
    e2e_s = float(np.min(ts[1:]))
    out["cfg3_predict"] = {"n_cells": int(data.n_cells), "n_ctp": int(data.n_ctp), "kernel_ms": kms,
                           "ctp_per_s": data.n_ctp / (kms * 1e-3), "flop_per_ctp": F_ALG_PREDICT,
                           "frac": data.n_ctp * F_ALG_PREDICT / (kms * 1e-3) / 1e12 / fp64_peak,
                           "e2e_ms": e2e_s * 1e3, "e2e_ctp_per_s": data.n_ctp / e2e_s, "d2h_bytes": int(3 * 14 * 8 * data.n_ctp),
                           "what": "forward + backward + combine (strict kernels); e2e = ggp_predict14: host params in, all three outputs "
                                   "as 14 doubles per time point into pinned host memory"}
    # the north star's target line: ONE log-likelihood evaluation of this 1 M-cell forest, strict and fast (gate against strict,
    # which equals the oracle per cell), as a fraction of the FP64 peak
    tgt = {"n_cells": int(data.n_cells), "n_ctp": int(data.n_ctp)}
    lls = {}
    for mode in ("strict", "fast"):
        f.set_mode(mode)
        lls[mode] = float(ggp.total_likelihood(P[0], f))
        ms = []
        for _ in range(5):
            ggp.total_likelihood(P[0], f)
            ms.append(f.last_kernel_ms)
        k = float(np.median(ms))
        tgt[mode] = {"kernel_ms": k, "ctp_per_s": data.n_ctp / (k * 1e-3), "frac_algorithmic": data.n_ctp * F_ALG / (k * 1e-3) / 1e12 / fp64_peak,
                     "loglik": lls[mode]}
    tgt["fast"]["nodes"] = int(f.last_fast_nodes)
    tgt["fast"]["strict_reruns"] = int(f.last_strict_reruns)
    tgt["fast_vs_strict_rel"] = abs(lls["fast"] - lls["strict"]) / abs(lls["strict"])
    out["target_1m_cells_loglik"] = tgt
    f.close()
    del pins
    # configs[3]: a 256-vector slice of the 4096-vector scan over the configs[1] forest, one ggp_loglik call, fresh mode
    data = ggp.simulate_forest(10000, 6, seed=20261018)
    f = ggp.Forest(data, device=device)
    vecs = np.tile(ggp.PARAMS_CONST_GAUSS, (256, 1))
    for k in range(256):
        vecs[k, k % 11] *= 0.8 + 0.4 * (k // 11) / 23.0
    cfg4 = {"n_vec": 256, "n_ctp": int(data.n_ctp)}
    for mode in ("strict", "fast"):
        f.set_mode(mode)
        ggp.total_likelihood(vecs[:8], f, raise_on_nan=False)
        t0 = time.perf_counter()
        ll = ggp.total_likelihood(vecs, f, raise_on_nan=False)
        dt = time.perf_counter() - t0
        cfg4[mode] = {"evals_per_s": 256 / dt, "ctp_per_s": 256 * data.n_ctp / dt, "kernel_ms": f.last_kernel_ms,
                      "frac": 256 * data.n_ctp * F_ALG / (f.last_kernel_ms * 1e-3) / 1e12 / fp64_peak, "finite": int(np.isfinite(ll).sum()),
                      "strict_reruns": int(f.last_strict_reruns)}
    out["cfg4_scan_slice"] = cfg4
    f.close()
    # configs[4]: -j on a 100 k-cell forest with two segments, tol 1e-10
    P2 = np.stack([ggp.PARAMS_SCALED_BINOMIAL, ggp.PARAMS_SCALED_BINOMIAL * np.array([1, 1, 1, 2, 1, 1, 1, 1, 1, 1, 1.])])
    data = ggp.simulate_forest(1587, 6, params=ggp.PARAMS_SCALED_BINOMIAL, noise_model="scaled", division_model="binomial",
                               seed=20261018, n_segments=2)
    f = ggp.Forest(data, device=device)
    ggp.prediction_forward_backward(f, P2, forward=False, backward=False, combined=False)
    ggp.count_joints(f, P2, 1e-10, 0, 1000)          # per-point preparation (cached on the handle)
    prep_ms = f.last_kernel_ms
    n_j, walk = 0, []
    for _ in range(2):
        n_j = ggp.count_joints(f, P2, 1e-10)
        walk.append(f.last_kernel_ms)
    rows = 100000
    n_rec = ggp.count_joints(f, P2, 1e-10, 0, rows)
    pin_rec = (torch.empty(n_rec, dtype=torch.int64).pin_memory().numpy(), torch.empty(n_rec, dtype=torch.int64).pin_memory().numpy(),
               torch.empty((n_rec, 44), dtype=torch.float64).pin_memory().numpy())
    rec_ts = []
    for _ in range(2):
        t0 = time.perf_counter()
        r, c, m, v = ggp.collect_joint_distributions(f, P2, 1e-10, row_begin=0, row_end=rows, out=pin_rec)
        rec_ts.append(time.perf_counter() - t0)
    rec_s = float(np.min(rec_ts))
    ts = []
    for _ in range(2):
        t0 = time.perf_counter()
        sums, nj2 = ggp.api.correlation_sums(f, P2, 15.0, 200)
        ts.append(time.perf_counter() - t0)
    out["cfg5_joints"] = {"n_cells": int(data.n_cells), "n_ctp": int(data.n_ctp), "joints": int(n_j), "prep_ms": prep_ms,
                          "reduced_ms": float(np.min(ts)) * 1e3, "reduced_joints_per_s": nj2 / float(np.min(ts)),
                          "reduced_what": "ggp_correlation_sums: walk + lag-binned moment sums of the correlation functions (200 lags) on the "
                                          "device, 80 kB of sums to the host, no record leaves the GPU",
                          "walk_ms": float(np.min(walk)), "joints_per_s": n_j / (np.min(walk) * 1e-3), "flop_per_joint": F_ALG_JOINT,
                          "frac": n_j * F_ALG_JOINT / (np.min(walk) * 1e-3) / 1e12 / fp64_peak,
                          "records_per_s": len(r) / rec_s, "records": int(len(r)),
                          "what": "every start point, count only (walk); records_per_s = the first %d start points with their records sorted "
                                  "on the device and copied into pinned host arrays (368 B per record)" % rows}
    f.close()
    out["cfg1_example"] = measure_example(ggp)
    return out


def measure_example(ggp):
    """BASELINE configs[0], the reference's own example data set (one tree, 13 generations, 22 065 points; fixture
    tests/golden/example_forest.npz): latency of one evaluation and of a 400-vector batch, and the command line's -m -p in the fast
    mode (binary forest file in; the reference documents "around 5 min" for this run)"""
    try:
        z = np.load(os.path.join(ROOT, "tests", "golden", "example_forest.npz"))
        data = ggp.LineageData(cell_offset=z["cell_offset"], parent=z["parent"], time=z["time"], log_length=z["log_length"], fp=z["fp"],
                               noise_model="scaled", division_model="binomial")
        P = np.asarray(z["params"], dtype=np.float64)
        f = ggp.Forest(data)
        res = {"n_ctp": int(data.n_ctp), "n_cells": int(data.n_cells), "generations": int(f.n_generations)}
        for mode in ("strict", "fast"):
            f.set_mode(mode)
            for n_vec in (1, 400):
                vecs = np.tile(P, (n_vec, 1))
                ggp.total_likelihood(vecs, f)
                ts = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    ggp.total_likelihood(vecs, f)
                    ts.append(time.perf_counter() - t0)
                res["%s_ms_%d_vec" % (mode, n_vec)] = float(np.median(ts)) * 1e3
        f.close()
        from gfp_gaussian_process_b200 import io
        cli = os.path.join(ROOT, "gfp_gaussian_process_b200", "bin", "gfp_gaussian")
        with tempfile.TemporaryDirectory() as tmp:
            io.write_forest_binary(os.path.join(tmp, "example.ggpf"), data)
            open(os.path.join(tmp, "cfg.txt"), "w").write("fp_auto = 0\n")
            with open(os.path.join(tmp, "p.txt"), "w") as fh:   # everything free except beta, like the example's parameter file
                for i, (name, v) in enumerate(zip(ggp.PARAM_NAMES, P)):
                    fh.write("%s = %r\n" % (name, float(v)) if i == 6 else "%s = %r, %r\n" % (name, float(v), float(v) * 0.1))
            t0 = time.perf_counter()
            r = subprocess.run(["timeout", "300", cli, "-i", os.path.join(tmp, "example.ggpf"), "-b", os.path.join(tmp, "p.txt"), "-c",
                                os.path.join(tmp, "cfg.txt"), "-m", "-p", "--fast", "-o", os.path.join(tmp, "out")], capture_output=True, text=True)
            res["cli_minimize_predict_fast_s"] = time.perf_counter() - t0
            res["cli_rc"] = r.returncode
            logs = [x for x in os.listdir(os.path.join(tmp, "out")) if x.endswith(".log")] if os.path.isdir(os.path.join(tmp, "out")) else []
            if logs:
                text = open(os.path.join(tmp, "out", logs[0])).read()
                res["cli_log"] = [ln for ln in text.split("\n") if ln.startswith("Stopped") or ln.startswith("Found maximum")]
        return res
    except Exception as e:   # an extra of the bench line: never lose the line over it
        return {"error": repr(e)}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
