#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 pairwise-distance engine (contract: task statement).

N = 1 : one step = raft_b200.distance.pairwise_distance L2Expanded 100000 x 100000 x 128 fp32
        (BASELINE.json configs[1]; operand prep + tcgen05 kernel), inputs resident in HBM.
        After the timed region the result of the last step is CHECKED (fp64 re-evaluation of sampled pairs on
        the device, oracle/device_check.py -> "parity"), the GPU baselines are timed on the same shapes in the
        same process ("gpu_baselines": cuBLASLt-SGEMM composition of the reference's surviving primitives,
        torch.cdist, a runtime probe for pylibraft / cuvs), and the other BASELINE configs are timed + checked.
N > 1 : one step = fusedL2NN 1,000,000 queries x 8,000,000 db rows x 96 (configs[3]); the db is
        row-sharded over the ranks, packed min-loc all-reduces (NCCL, int64 MIN).  Strong scaling: total work
        fixed.  Rank 0 first runs the SAME job un-sharded on its own GPU (same session, same data), so every
        line carries "scaling": {t1_ms, tN_ms, speedup, efficiency}; every rank checks the reduced result
        against the exact fp64 arg-min over its own shard (combined across ranks) -> "parity".
--impl reference : the CPU restatement (oracle port: numpy expanded form on multithreaded BLAS,
        all host cores) on a bounded sample of the same workload.  The reference's own kernels for
        this path are not in the reference snapshot (SURVEY.md section 0), so there is nothing else to run.
--dump-outputs DIR : after the timed steps, what the last timed step returned is written as DIR/<name>.npy
        (float32 / float64, 32 MB at N = 1, 12 MB at N > 1), so that two builds run with the same arguments
        (same seeded inputs) can be compared output for output:
          N = 1 : pairwise_distance.npy -- the [2048, 4096] float32 sub-matrix of the 100000 x 100000 result at
                  rows / columns drawn by torch.randperm with seed 5 (sorted), see DUMP_SAMPLE
          N > 1 : fused_l2_nn_idx.npy (float64, exact) and fused_l2_nn_val.npy (float32), all 1M queries (rank 0)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAIRWISE = dict(m=100_000, n=100_000, k=128)
FUSED_NN = dict(m=1_000_000, n=8_000_000, k=96)
METRIC = "distance-pairs/sec"
DUMP_SAMPLE = dict(rows=2048, cols=4096, seed=5)   # --dump-outputs at N = 1: the full result is 40 GB


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def ncu_traffic(name):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    for f in ("r02_traffic.json", "r01_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", f)))[name]
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def blobs_device(rows, cols, seed, centers, torch, device):
    """make_blobs-like data on the device: 5 centres ~U[-10,10]^k, sigma 1 (SURVEY.md 8(d))."""
    g = torch.Generator(device=device).manual_seed(seed)
    lab = torch.randint(0, centers.shape[0], (rows,), device=device, generator=g)
    out = torch.randn(rows, cols, device=device, generator=g)
    out += centers[lab]
    return out


def centers_device(cols, torch, device):
    g = torch.Generator(device=device).manual_seed(42)
    return torch.rand(5, cols, device=device, generator=g) * 20.0 - 10.0


# ------------------------------------------------------------------------------------------------
def cpu_l2_expanded_numpy(x, y, out=None):
    """oracle port, 'reference-style' composition on host cores: row norms + SGEMM + epilogue."""
    import numpy as np
    xn = np.einsum("ij,ij->i", x, x)
    yn = np.einsum("ij,ij->i", y, y)
    d = x @ y.T
    d *= -2.0
    d += xn[:, None]
    d += yn[None, :]
    np.maximum(d, 0.0, out=d)
    return d


def cpu_fused_nn_numpy(x, y, block=16384):
    import numpy as np
    xn = np.einsum("ij,ij->i", x, x)
    best = np.full(x.shape[0], np.inf, np.float32)
    idx = np.zeros(x.shape[0], np.int64)
    for j0 in range(0, y.shape[0], block):
        yb = y[j0:j0 + block]
        d = -2.0 * (x @ yb.T) + np.einsum("ij,ij->i", yb, yb)[None, :]
        loc = d.argmin(axis=1)
        v = d[np.arange(len(x)), loc]
        upd = v < best
        best[upd] = v[upd]
        idx[upd] = loc[upd] + j0
    return idx, np.maximum(best + xn, 0)


def cpu_baseline(workload, seconds_budget=12.0, reps_fixed=None, warm=1):
    """Times the CPU port on a bounded sample of the workload; returns the cpu_baseline object."""
    import numpy as np
    import oracle  # noqa: F401  (the port lives in oracle/: allowed here, see task statement (4))
    cores = os.cpu_count() or 1
    if workload == "pairwise":
        k, rows = PAIRWISE["k"], 8192
        x, _, c = oracle.make_blobs(rows, k, seed=1234)
        y, _, _ = oracle.make_blobs(rows, k, seed=4321, centers=c)
        fn, pairs = (lambda: cpu_l2_expanded_numpy(x, y)), rows * rows
        sample = f"L2Expanded {rows}x{rows}x{k} fp32 slice of the 100000x100000x128 job, numpy/OpenBLAS"
    else:
        k, m, n = FUSED_NN["k"], 8192, 65536
        x, _, c = oracle.make_blobs(m, k, seed=1234)
        y, _, _ = oracle.make_blobs(n, k, seed=4321, centers=c)
        fn, pairs = (lambda: cpu_fused_nn_numpy(x, y)), m * n
        sample = f"fusedL2NN {m}x{n}x{k} fp32 slice of the 1Mx8Mx96 job, numpy/OpenBLAS"
    for _ in range(max(1, warm)):
        fn()
    t0, reps = time.perf_counter(), 0
    while True:
        fn()
        reps += 1
        if reps_fixed is not None:
            if reps >= reps_fixed:
                break
        elif time.perf_counter() - t0 > seconds_budget or reps >= 50:
            break
    dt = (time.perf_counter() - t0) / reps
    return {"value": pairs / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": sample + f", {reps} reps of {dt:.3f} s"}, dt, pairs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = "pairwise" if args.gpus == 1 else "fused_l2_nn"
    # each step = one pass over the bounded sample
    cb, dt, pairs = cpu_baseline(workload, reps_fixed=max(1, args.steps), warm=max(1, args.warmup))
    cfg = ({"workload": "pairwise_distance L2Expanded 100000x100000x128 fp32 -> fp32 [m,n]",
            "sample_per_step": "8192x8192x128 slice (bounded so the run ends in minutes)"}
           if workload == "pairwise" else
           {"workload": "fusedL2NN 1000000 queries x 8000000 db x 96 fp32, db row-sharded",
            "sample_per_step": "8192x65536x96 slice (bounded so the run ends in minutes)"})
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic make_blobs-like (5 centres U[-10,10], sigma 1)", "config": cfg,
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference kernels for this path are absent from the reference snapshot; this arm is the CPU oracle port"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def time_steps(fn, steps, warmup, torch, sync_all=None):
    for _ in range(warmup):
        fn()
    if sync_all:
        sync_all()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    if sync_all:
        sync_all()
    per = [a.elapsed_time(b) for a, b in ev]
    total = ev[0][0].elapsed_time(ev[-1][1])
    return total / steps, per


def dump_outputs(dirname, arrays):
    """--dump-outputs: {name: tensor} -> dirname/<name>.npy; integer outputs as float64 (exact below 2^53)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype.kind in "iu" or a.dtype == np.float64 else np.float32)
        np.save(os.path.join(dirname, name + ".npy"), a)


def pairwise_dump_sample(out, torch):
    """The fixed DUMP_SAMPLE sub-matrix of a pairwise result (sorted seeded rows x sorted seeded columns)."""
    g = torch.Generator(device=out.device).manual_seed(DUMP_SAMPLE["seed"])
    rows = torch.randperm(out.shape[0], device=out.device, generator=g)[:DUMP_SAMPLE["rows"]].sort().values
    cols = torch.randperm(out.shape[1], device=out.device, generator=g)[:DUMP_SAMPLE["cols"]].sort().values
    return out[rows[:, None], cols[None, :]]


def gpu_baselines_pairwise(x, y, out, m, n, k, ours_ms, torch, steps=5, warm=2):
    """GPU baselines for configs[1] (L2Expanded m x n x k fp32), timed like the engine (CUDA events, output buffer
    reused; every step streams 40+ GB through the 126 MB L2, so nothing is cached between steps)."""
    import baseline
    res = {}
    dev = x.device
    # (i) what the reference's surviving primitives compose to (baseline/gpu_composition.cu)
    try:
        L = baseline.lib()
        baseline.check(L.bl_init())
        xn = torch.empty(m, device=dev)
        yn = torch.empty(n, device=dev)
        ws = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        fn = lambda: baseline.check(L.bl_pairwise_l2(st, out.data_ptr(), x.data_ptr(), y.data_ptr(), xn.data_ptr(),
                                                     yn.data_ptr(), m, n, k, 0, ws.data_ptr(), ws.numel()))
        ms, _ = time_steps(fn, steps, warm, torch)
        from oracle import device_check as dc
        par = dc.check_pairwise_sampled(out, x, y, 0, count=50_000, eps=1e-4)
        res["cublaslt_sgemm_composition"] = {
            "ms": ms, "pairs_per_s": m * n / (ms * 1e-3),
            "what": "row norms + cublasLtMatmul fp32 (CUBLAS_COMPUTE_32F, no TF32) + one elementwise pass: the composition "
                    "of raft::linalg::norm / gemm / map_offset (cublaslt_wrappers.hpp:35-38,268-313) -- 3 passes over m x n",
            "parity_vs_fp64": par, "speedup_of_engine": ms / ours_ms}
        del xn, yn, ws
    except Exception as e:  # noqa: BLE001
        res["cublaslt_sgemm_composition"] = {"unavailable": repr(e)[:200]}
    # (ii) torch.cdist (cuBLAS SGEMM path, TF32 off = torch default) -- needs its own 40 GB result (+ temporaries)
    try:
        torch.backends.cuda.matmul.allow_tf32 = False
        fn = lambda: torch.cdist(x, y, p=2.0, compute_mode="use_mm_for_euclid_dist")
        ms, _ = time_steps(fn, 3, 1, torch)
        res["torch_cdist"] = {"ms": ms, "pairs_per_s": m * n / (ms * 1e-3), "speedup_of_engine": ms / ours_ms,
                              "what": "torch.cdist(p=2, use_mm_for_euclid_dist): euclidean (sqrt) distances, allocates its own output"}
    except Exception as e:  # noqa: BLE001
        res["torch_cdist"] = {"unavailable": repr(e)[:200]}
    torch.cuda.empty_cache()
    # (iii) the reference's own GPU kernels, if some RAFT <= 25.12 / cuVS wheel is importable on this box
    probe = {}
    for mod in ("pylibraft.distance", "cuvs.distance"):
        try:
            mobj = __import__(mod, fromlist=["x"])
            where = os.path.abspath(getattr(mobj, "__file__", "") or "")
            if where.startswith(ROOT):
                probe[mod] = "only this repo's alias package (no RAFT / cuVS wheel on the box)"
            else:
                probe[mod] = "importable at " + where + " (not timed: unexpected on this image)"
        except Exception as e:  # noqa: BLE001
            probe[mod] = "not importable: " + type(e).__name__
    res["reference_gpu_kernels_probe"] = probe
    return res


def gpu_baseline_nn_sample(q, db, ours_pairs_per_s, torch, mq=65536, nd=1 << 20, chunk=131072):
    """fusedL2NN by composition (SGEMM + elementwise + row arg-min per db chunk, baseline/gpu_composition.cu) on a
    bounded sample of the 1M x 8M job: mq queries x nd db rows; the rate is per pair, the full job is 122x the sample."""
    import baseline
    try:
        L = baseline.lib()
        dev = q.device
        k = q.shape[1]
        xs, ys = q[:mq].contiguous(), db[:nd].contiguous()
        tile = torch.empty((mq, chunk), dtype=torch.float32, device=dev)
        xn, yn = torch.empty(mq, device=dev), torch.empty(chunk, device=dev)
        bv, bi = torch.empty(mq, device=dev), torch.empty(mq, dtype=torch.int32, device=dev)
        ws = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        fn = lambda: baseline.check(L.bl_l2_nn(st, bv.data_ptr(), bi.data_ptr(), xs.data_ptr(), ys.data_ptr(), tile.data_ptr(),
                                               xn.data_ptr(), yn.data_ptr(), mq, nd, k, chunk, ws.data_ptr(), ws.numel()))
        ms, _ = time_steps(fn, 3, 1, torch)
        rate = mq * nd / (ms * 1e-3)
        return {"ms_sample": ms, "sample": f"{mq} queries x {nd} db rows x {k} (chunks of {chunk} db rows), extrapolated per pair",
                "pairs_per_s": rate, "speedup_of_engine": ours_pairs_per_s / rate,
                "what": "cublasLt SGEMM (CUBLAS_COMPUTE_32F) + elementwise pass + row arg-min pass per chunk, merged across chunks"}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)[:200]}


def nn_parity_1gpu(idx, val, q, db, torch, sample=16384, seed=3):
    from oracle import device_check as dc
    g = torch.Generator(device=q.device).manual_seed(seed)
    rows = torch.randperm(q.shape[0], device=q.device, generator=g)[:sample]
    ref_val, ref_idx = dc.nn_exact_fp64(q[rows], db)
    r = dc.check_nn(idx[rows], val[rows], ref_val, ref_idx, q[rows], lambda ix: db[ix])
    r["what"] = f"{sample} sampled queries vs the exact fp64 arg-min over all {db.shape[0]} db rows"
    return r


def run_pairwise_1gpu(args):
    import numpy as np
    import torch
    from oracle import device_check as dc
    from raft_b200.common import DeviceResources
    from raft_b200.distance import HostPairwise, fused_l2_nn, pairwise_distance
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peaks, peak_src = measured_peaks()
    m, n, k = PAIRWISE["m"], PAIRWISE["n"], PAIRWISE["k"]
    c = centers_device(k, torch, dev)
    x = blobs_device(m, k, 1234, c, torch, dev)
    y = blobs_device(n, k, 4321, c, torch, dev)
    out = torch.empty((m, n), dtype=torch.float32, device=dev)
    h = DeviceResources()
    fn = lambda: pairwise_distance(x, y, out=out, metric="sqeuclidean", handle=h)
    # the dominant kernel's own launch durations, from CUDA events the library records on the launching
    # stream around expanded_tc_kernel during the timed steps (no synchronisation until the region ends)
    import ctypes
    from raft_b200 import _lib
    L = _lib.lib()
    state = {"n": 0}

    def fn_counted():
        state["n"] += 1
        if state["n"] == args.warmup + 1:          # first timed step
            _lib.check(L.b2d_profile_begin(max(1, args.steps)))
        fn()
    out.fill_(float("nan"))
    with ClockSampler(0) as cs:
        ms, per = time_steps(fn_counted, args.steps, args.warmup, torch)
    kbuf = (ctypes.c_float * max(1, args.steps))()
    kcnt = ctypes.c_int(0)
    _lib.check(L.b2d_profile_end(kbuf, max(1, args.steps), ctypes.byref(kcnt)))
    kernel_ms = [float(kbuf[i]) for i in range(kcnt.value)]
    k_ms = sum(kernel_ms) / len(kernel_ms) if kernel_ms else ms
    clocks = cs.summary()
    pairs = m * n
    if args.dump_outputs:            # before the other configs below reuse `out`
        dump_outputs(args.dump_outputs, {"pairwise_distance": pairwise_dump_sample(out, torch)})
    # ---- parity of what was just timed: the result of the last timed step, re-evaluated in fp64 on the device
    parity = dc.check_pairwise_sampled(out, x, y, 0, count=200_000, eps=1e-4)
    parity["what"] = "L2Expanded 100000x100000x128: sampled pairs incl. tile corners / matrix edges vs fp64, CompareApprox(1e-4)"
    parity["every_tile_written"] = bool(torch.isfinite(out[::127, ::251]).all().item())
    alg_bytes = 4 * (m * k + n * k) + 4 * m * n
    roof = {"bound": "hbm", "achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "peak_source": f"{peak_src} (MEASURED_PEAKS.json hbm_gbs, copy read+write)",
            "kernel": "expanded_tc_kernel (tcgen05, EPI_STORE): mean launch duration over the timed steps, CUDA events "
                      "on the launching stream (b2d_profile_begin/end)",
            "kernel_ms": k_ms, "launches_timed": len(kernel_ms),
            "whole_step": {"achieved": alg_bytes / (ms * 1e-3) / 1e9, "frac": alg_bytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                           "note": "the same bytes over the whole step, i.e. incl. the two operand-prep launches"},
            "traffic": ncu_traffic("pairwise_100k")}
    roof["frac"] = roof["achieved"] / roof["peak"]
    # ---- GPU baselines on the same shapes, same process, same timing method
    gpu_bl = gpu_baselines_pairwise(x, y, out, m, n, k, ms, torch)
    # ---- the other BASELINE.json configs, timed briefly in the same run AND checked (sampled fp64 re-evaluation)
    others = {}

    def t_ms(f, steps=3, warm=1):
        ms_, _ = time_steps(f, steps, warm, torch)
        return ms_

    def chk(o, xs, ys, metric, count=100_000, row_offset=0):
        r = dc.check_pairwise_sampled(o, xs, ys, metric, count=count, eps=1e-4, row_offset=row_offset)
        return {"checked": r["checked"], "n_bad": r["n_bad"], "max_rel_err": r["max_rel_err"]}
    for metric, mt in (("cosine", 2), ("correlation", 10)):
        ms_o = t_ms(lambda: pairwise_distance(x, y, out=out, metric=metric, handle=h))
        others[f"{metric} 100000x100000x128 f32"] = {"ms": ms_o, "pairs_per_s": pairs / (ms_o * 1e-3),
                                                     "hbm_gbs": alg_bytes / (ms_o * 1e-3) / 1e9, "parity": chk(out, x, y, mt)}
    m3, k3 = 50_000, 256
    c3 = centers_device(k3, torch, dev)
    x3 = blobs_device(m3, k3, 1234, c3, torch, dev)
    y3 = blobs_device(m3, k3, 4321, c3, torch, dev)
    out3 = out.view(-1)[: m3 * m3].view(m3, m3)
    for metric, name, mt in (("cityblock", "L1", 3), ("sqeuclidean_unexpanded", "L2Unexpanded", 4), ("chebyshev", "Linf", 7)):
        ms_o = t_ms(lambda: pairwise_distance(x3, y3, out=out3, metric=metric, handle=h), steps=2)
        others[f"{name} 50000x50000x256 f32"] = {
            "ms": ms_o, "pairs_per_s": m3 * m3 / (ms_o * 1e-3),
            "hbm_gbs": (8.0 * m3 * k3 + 4.0 * m3 * m3) / (ms_o * 1e-3) / 1e9,
            "fp32_lane_ops_per_s": 2.0 * m3 * m3 * k3 / (ms_o * 1e-3), "bound": "fp32 pipe (148 SMs x 128 lanes x clk)",
            "parity": chk(out3, x3, y3, mt)}
    del x3, y3
    # fused brute-force kNN (SURVEY.md 8(f2)): top-16 of every row of the 100000x100000x128 problem, matrix never written
    from raft_b200.neighbors import brute_force
    ms_o = t_ms(lambda: brute_force.knn(y, x, k=16, handle=h), steps=2)
    others["kNN k=16 100000x100000x128 f32 (fused select)"] = {"ms": ms_o, "pairs_per_s": pairs / (ms_o * 1e-3)}
    # fp16-in / fp32-accumulate 200000x200000x64: the 160 GB result is produced in 4 row blocks into a reused buffer
    m5, k5, blk = 200_000, 64, 50_000
    c5 = centers_device(k5, torch, dev)
    x5 = blobs_device(m5, k5, 1234, c5, torch, dev).half()
    y5 = blobs_device(m5, k5, 4321, c5, torch, dev).half()
    out5 = out.view(-1)[: blk * m5].view(blk, m5)

    def fp16_pass():
        for r0 in range(0, m5, blk):
            pairwise_distance(x5[r0:r0 + blk], y5, out=out5, metric="sqeuclidean", handle=h)
    ms_o = t_ms(fp16_pass, steps=2)
    others["L2Expanded 200000x200000x64 f16-in/f32-acc (4 row blocks, reused 40 GB buffer)"] = {
        "ms": ms_o, "pairs_per_s": float(m5) * m5 / (ms_o * 1e-3), "hbm_gbs": 4.0 * m5 * m5 / (ms_o * 1e-3) / 1e9,
        "parity": dict(chk(out5, x5, y5, 0, row_offset=m5 - blk), note="last row block, vs the fp16-rounded inputs")}
    del x5, y5, out5, out3
    del out
    torch.cuda.empty_cache()

    # ---- e2e: host buffers in, result streamed back to pinned host memory, per step
    xh, yh = x.cpu().numpy(), y.cpu().numpy()
    hp = HostPairwise(m, n, k)
    e2e_steps = max(1, min(args.steps, 3))
    hp.run(xh, yh, metric="sqeuclidean")          # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hp.run(xh, yh, metric="sqeuclidean")
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e = {"value": pairs / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": hp.h2d_bytes,
           "d2h_bytes_per_step": hp.d2h_bytes, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
           "path": "raft_b200.distance.HostPairwise.run: pinned H2D of X,Y; ~1 GiB row slabs; D2H of every slab "
                   "into pinned host memory overlapped with the next slab's kernel"}
    del hp
    torch.cuda.empty_cache()

    # ---- 1-GPU fusedL2NN (configs[3] on one GPU): timed, checked, and the composition baseline beside it
    fm, fn_, fk = FUSED_NN["m"], FUSED_NN["n"], FUSED_NN["k"]
    c2 = centers_device(fk, torch, dev)
    q = blobs_device(fm, fk, 1234, c2, torch, dev)
    db = torch.cat([blobs_device(hi - lo, fk, 4321 + r, c2, torch, dev) for r, (lo, hi) in
                    enumerate([(fn_ * r // 8, fn_ * (r + 1) // 8) for r in range(8)])])   # the 8-rank job's database
    nn_steps = max(1, min(args.steps, 2))
    res = {}

    def nn_step():
        res["iv"] = fused_l2_nn(q, db, sqrt=False, handle=h)
    nn_ms, _ = time_steps(nn_step, nn_steps, 1, torch)
    nn = {"workload": "fusedL2NN 1000000x8000000x96 fp32, 1 GPU", "value": fm * fn_ / (nn_ms * 1e-3),
          "unit": "pairs/s", "ms_per_step": nn_ms, "steps": nn_steps,
          "roofline": {"bound": "tensor", "achieved": 2.0 * fm * fn_ * fk / (nn_ms * 1e-3) / 1e12,
                       "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                       "note": "algorithmic 2mnk FLOP / time.  The exact kernel executes 3x that on the tensor pipe "
                               "(fp32-grade 3-term fp16 split); the screened search (1M-row chunks of the db: exact on "
                               "1/32 of the blocks, 1-product screen on the rest, exact re-evaluation of the candidates) "
                               "executes ~1.06x"}}
    nn["roofline"]["frac"] = nn["roofline"]["achieved"] / nn["roofline"]["peak"]
    nn["parity"] = nn_parity_1gpu(res["iv"][0], res["iv"][1], q, db, torch)
    nn["gpu_baseline_composition"] = gpu_baseline_nn_sample(q, db, nn["value"], torch)
    del q, db

    cb, _, _ = cpu_baseline("pairwise", seconds_budget=10.0)
    line = {"metric": METRIC, "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32",
            "data": "synthetic make_blobs-like (5 centres U[-10,10]^k, sigma 1, seeds 1234/4321), generated on device",
            "config": {"workload": "pairwise_distance L2Expanded 100000x100000x128 fp32 -> fp32 [m,n]",
                       "precision": "fp32-grade: 3-term fp16 hi/lo split, fp32 accumulate in TMEM",
                       "l2": "every step streams 40 GB of output through the 126 MB L2 (no reuse across steps)"},
            "roofline": roof, "parity": parity, "gpu_baselines": gpu_bl, "cpu_baseline": cb, "e2e": e2e,
            "gpu_launches": 3 * args.steps, "clocks": clocks, "fused_l2_nn": nn, "other_configs": others,
            "ms_per_step_all": [round(v, 4) for v in per]}
    print(json.dumps(line))


def nn_launches(shard_rows, world):
    """Kernels of this repo per sharded fusedL2NN call (api.cu fused_nn_keys): per b2d_fused_l2_nn_keys call and
    1M-row chunk: 2 prep + exact sample + seed + trial screen + decide + main screen + decide + candidate
    re-evaluation + 2 conditional exact passes = 11; + key init + finalize."""
    from raft_b200.distance.fused_l2_nn import plan_exchanges
    calls = plan_exchanges(shard_rows, world)   # (shard_rows: n_total // world)
    chunks = lambda n: max(1, -(-n // (1 << 20)))
    return 11 * sum(chunks(c) for c in calls) + 2


def run_fused_nn_multi(args):
    import torch
    import torch.distributed as dist
    from oracle import device_check as dc
    from raft_b200.common import DeviceResources
    from raft_b200.distance import fused_l2_nn, fused_l2_nn_sharded, shard_bounds
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    # NCCL writes its version banner (and any NCCL_DEBUG output) to the C-level stdout: park fd 1 on stderr for
    # the whole run and write the single JSON line to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks, peak_src = measured_peaks()
    m, n, k = FUSED_NN["m"], FUSED_NN["n"], FUSED_NN["k"]
    c = centers_device(k, torch, dev)
    q = blobs_device(m, k, 1234, c, torch, dev)                 # queries replicated (same seed on every rank)
    lo, hi = shard_bounds(n, world, rank)
    # the database is defined by its 8 row blocks (seed 4321 + block): a rank generates the blocks of its shard, so the
    # 1-, 2-, 4- and 8-GPU runs (and rank 0's un-sharded base run below) all search the SAME 8M rows
    blocks = [(n * r // 8, n * (r + 1) // 8) for r in range(8)]

    def db_rows(a, b):
        parts = []
        for r, (blo, bhi) in enumerate(blocks):
            s0, s1 = max(a, blo), min(b, bhi)
            if s0 < s1:
                blk = blobs_device(bhi - blo, k, 4321 + r, c, torch, dev)
                parts.append(blk[s0 - blo:s1 - blo])
        return torch.cat(parts) if len(parts) > 1 else parts[0].contiguous()
    h = DeviceResources()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- same-session 1-GPU base of the scaling record: rank 0 runs the whole job un-sharded (others wait)
    t1_ms, base = None, None
    if rank == 0:
        full = db_rows(0, n)
        r1 = {}

        def base_step():
            r1["iv"] = fused_l2_nn(q, full, sqrt=False, handle=h)
        t1_ms, _ = time_steps(base_step, 2, 1, torch)
        base = (r1["iv"][0].clone(), r1["iv"][1].clone())
        del full, r1
        torch.cuda.empty_cache()
    sync_all()
    db = db_rows(lo, hi)                                        # this rank's row block of the database
    keys = torch.empty(m, dtype=torch.int64, device=dev)
    last = {}

    def step():
        last["iv"] = fused_l2_nn_sharded(q, db, lo, sqrt=False, handle=h, keys=keys, n_total=n)

    with ClockSampler(local) as cs:
        ms, per = time_steps(step, args.steps, args.warmup, torch, sync_all=sync_all)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"fused_l2_nn_idx": last["iv"][0], "fused_l2_nn_val": last["iv"][1]})
    # ---- parity on EVERY rank: the reduced result vs the exact fp64 arg-min (own shard, combined across ranks)
    g = torch.Generator(device=dev).manual_seed(3)
    rows = torch.randperm(m, device=dev, generator=g)[:8192]
    lv, la = dc.nn_exact_fp64(q[rows], db, idx_offset=lo)       # exact over this shard, GLOBAL indices
    if world > 1:
        allv = [torch.empty_like(lv) for _ in range(world)]
        alla = [torch.empty_like(la) for _ in range(world)]
        dist.all_gather(allv, lv)
        dist.all_gather(alla, la)
        V, A = torch.stack(allv), torch.stack(alla)
        gv = V.min(dim=0).values
        ga = torch.where(V == gv[None, :], A, torch.full_like(A, 2 ** 62)).min(dim=0).values   # ties -> smaller index
    else:
        gv, ga = lv, la
    gi, gval = last["iv"][0][rows], last["iv"][1][rows]
    # fp64 distance of the row the engine chose: computed by the rank that owns it, summed across ranks
    own = (gi.long() >= lo) & (gi.long() < hi)
    dsel = torch.zeros(rows.numel(), dtype=torch.float64, device=dev)
    if int(own.sum()):
        dsel[own] = ((q[rows[own]].double() - db[gi.long()[own] - lo].double()) ** 2).sum(1)
    if world > 1:
        dist.all_reduce(dsel)
    same = gi.long() == ga
    gap = (dsel - gv).abs() / gv.clamp_min(1e-300)
    n_bad_val, max_rel = dc.compare_approx(gval, gv, 1e-4)
    par = torch.tensor([float(same.float().mean()), float((same | (gap <= 1e-6)).float().mean()), float(n_bad_val), max_rel],
                       dtype=torch.float64, device=dev)
    pmin, pmax = par.clone(), par.clone()
    if world > 1:
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
    parity = {"checked_per_rank": int(rows.numel()), "ranks": world,
              "idx_strict_match": float(pmin[0]), "idx_tie_aware_match": float(pmin[1]), "val_n_bad": int(pmax[2]),
              "val_max_rel_err": float(pmax[3]),
              "what": "every rank: 8192 sampled queries, reduced (idx, dist) vs the exact fp64 arg-min over all shards "
                      "(per-shard fp64 minima all_gathered); worst rank reported"}
    if rank == 0 and base is not None:
        bv, sv = base[1].double(), last["iv"][1].double()
        parity["sharded_equals_unsharded"] = {"idx_equal_frac": float((base[0] == last["iv"][0]).float().mean()),
                                              "val_equal_frac": float((base[1] == last["iv"][1]).float().mean()),
                                              # rows that differ are fp32 near-ties: two db rows whose direct fp32 distances
                                              # differ by rounding only (each run re-measures the finalists IT kept)
                                              "val_max_rel_diff": float(((bv - sv).abs() / torch.clamp(torch.maximum(bv, sv), min=1e-30)).max())}
    if rank == 0:
        pairs = m * n
        tf = 2.0 * m * n * k / (ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"] * world, "unit": "TFLOP/s",
                "peak_source": f"{peak_src} (MEASURED_PEAKS.json bf16_tflops_sustained x n_gpus)",
                "kernel": "screen_tc_kernel (tcgen05, 1-product screen) + expanded_tc_kernel (EPI_MINLOC, exact on 1/32 of "
                          "the db blocks and wherever screening is called off); algorithmic 2mnk FLOP / time",
                "traffic": ncu_traffic("screen_tc_per_launch")}
        roof["frac"] = roof["achieved"] / roof["peak"]
        cb, _, _ = cpu_baseline("fused_l2_nn", seconds_budget=8.0)
        from raft_b200.distance.fused_l2_nn import plan_exchanges
        n_calls = len(plan_exchanges(n // world, world))
        line = {"metric": METRIC, "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "scaling_record": {"t1_ms": t1_ms, "tN_ms": ms, "speedup": (t1_ms / ms) if t1_ms else None,
                                   "efficiency": (t1_ms / ms / world) if t1_ms else None,
                                   "note": "t1 = the same job un-sharded on rank 0's GPU, same session, same data"},
                "vs_baseline": None, "dtype": "f32",
                "data": "synthetic make_blobs-like (5 centres U[-10,10]^k, sigma 1), generated on device",
                "config": {"workload": "fusedL2NN 1000000 queries x 8000000 db x 96 fp32, db row-sharded",
                           "parallelism": f"db_shard{world}",
                           "exchange": f"{n_calls} x all_reduce(int64 MIN) of 1M packed (dist,idx) keys per step (bounds between sub-chunks of the shard, result at the end)",
                           "l2": "db shard + queries exceed L2 for world<=8 (>=768 MB per rank)"},
                "roofline": roof, "parity": parity, "cpu_baseline": cb,
                "e2e": None, "gpu_launches": nn_launches(n // world, world) * args.steps, "clocks": cs.summary(),
                "ms_per_step_all": [round(v, 3) for v in per]}
    # e2e needs every rank to take part in the collective
    qh = q.cpu().pin_memory()
    dbh = db.cpu().pin_memory()

    def e2e_step():
        with torch.cuda.stream(h.torch_stream):
            q.copy_(qh, non_blocking=True)
            db.copy_(dbh, non_blocking=True)
        i, v = fused_l2_nn_sharded(q, db, lo, sqrt=False, handle=h, keys=keys, n_total=n)
        return i.cpu(), v.cpu()

    e2e_step()
    sync_all()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        e2e_step()
    sync_all()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    t = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        line["e2e"] = {"value": m * n / float(t.item()), "unit": "pairs/s",
                       "h2d_bytes_per_step": 4 * k * (m + (hi - lo)), "d2h_bytes_per_step": 8 * m,
                       "ms_per_step": float(t.item()) * 1e3, "steps": e2e_steps,
                       "path": "pinned H2D of queries + this rank's db shard, fused_l2_nn_sharded, D2H of (idx,dist)"}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus == 1 and world == 1:
        return run_pairwise_1gpu(args)
    return run_fused_nn_multi(args)


if __name__ == "__main__":
    main()
