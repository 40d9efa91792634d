#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native SpMV + Krylov hot path.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A "step" is one CSR SpMV  y = A x  of BASELINE.json configs[1]: random CSR fp64,
n = 10 000 000, nnz = 150 000 000 (15 distinct uniform columns per row), synthetic data from
workloads.py.  N > 1 (launched by torchrun, one rank per GPU): the matrix is split 1-D by
row ranges (strong scaling), every step all-gathers the x slices over NCCL and runs the local
SpMV; value = 2*nnz_total / max-over-ranks step time.

Printed JSON (one line, rank 0): metric / value / unit as BASELINE.json's metric, plus
  roofline     dominant kernel's algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json
  cpu_baseline the reference's own OMP executor (oracle/_ref) on this box's host cores,
               bounded sample of the same workload
  e2e          same metric through gko_b200::staged_apply with HOST buffers (H2D x, SpMV,
               D2H y every step; consecutive steps overlap on the copy streams)
  cg           CG iterations/s (cfg3 on 1 GPU, cfg5-style row-sharded on N GPUs)
`--impl reference` times the reference's CPU implementation only (no GPU work).
"""
import argparse
import json
import os
import sys
import threading
import time

# Thread binding of the CPU arm (the reference's OmpExecutor): must be in the environment BEFORE
# anything loads libgomp (numpy / torch do), otherwise it is ignored and the 64 threads float.
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import workloads as W  # noqa: E402

CFG = "cfg2"
N_ROWS = W.CONFIGS[CFG]["n"]
PER_ROW = W.CONFIGS[CFG]["per_row"]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """polls NVML (SM clock + clock-event reasons) every few ms during the timed region"""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, dev):
        self.samples, self.reasons, self.stop = [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(dev)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop and self.nv:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join()

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


class OutputDump:
    """--dump-outputs DIR: what every timed leg computed in its last step, as DIR/<name>.npy.  Each
    leg keeps a sample of its result vector at positions drawn by a seeded generator (the same in
    every run, 64 MB in all), so two builds run with the same arguments compare output for output."""
    MAX_BYTES = 64 << 20

    def __init__(self, path, world, stream):
        self.path, self.world, self.stream, self.arrays = path, world, stream, {}

    def take(self, name, local, r0, n_total, k):
        """local = rows [r0, r0 + local.numel()) of an n_total-row result; every rank calls this"""
        import torch
        import torch.distributed as dist
        k = min(k, n_total)
        idx = np.sort(np.random.default_rng(1).choice(n_total, k, replace=False))
        with torch.cuda.stream(self.stream):
            idx = torch.from_numpy(idx).to(local.device)
            mine = (idx >= r0) & (idx < r0 + local.numel())
            out = torch.zeros(k, dtype=local.dtype, device=local.device)
            out[mine] = local.reshape(-1)[idx[mine] - r0]
            if self.world > 1:  # each position is owned by one rank, the others add zeros
                dist.all_reduce(out)
            self.arrays[name] = out.cpu().numpy()

    def write(self):
        total = sum(a.nbytes for a in self.arrays.values())
        if total > self.MAX_BYTES:
            raise RuntimeError("--dump-outputs: %d bytes exceed %d" % (total, self.MAX_BYTES))
        os.makedirs(self.path, exist_ok=True)
        for name, a in self.arrays.items():
            np.save(os.path.join(self.path, name + ".npy"), a)


# ------------------------------------------------------------------ CPU arm (reference OMP)
def cfg2_on_host():
    """the FULL cfg2 matrix + x as numpy arrays (generated on the GPU when there is one: the
    counter-based hash of workloads.py gives the same bits on both, and 150 M entries take ~1 s there)"""
    try:
        import torch
        if torch.cuda.is_available():
            dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
            rp, ci, va = W.build(CFG, xp="torch", device=dev)
            x = W.vector(N_ROWS, xp="torch", device=dev)
            out = tuple(t.cpu().numpy() for t in (rp, ci, va, x))
            del rp, ci, va, x
            torch.cuda.empty_cache()
            return out
    except Exception:
        pass
    rp, ci, va = W.build(CFG, xp="np")
    return rp, ci, va, W.vector(N_ROWS)


def cpu_reference_spmv(mat, min_reps, min_seconds=2.0, reps=None):
    """the reference's OMP executor (oracle/_ref) on the full cfg2 -- same config as the GPU arm --
    or, if that was not built, the oracle port.  Reference methodology (benchmark/utils/timer):
    warm-up, then >= min_reps repetitions and >= min_seconds; exactly `reps` repetitions when given."""
    rp, ci, va, x = mat
    nnz = len(va)
    n = len(rp) - 1
    from oracle import ref
    if ref.available():
        cores = ref.use_physical_cores()
        _, sec1 = ref.spmv("csr", rp, ci, va, x, N_ROWS, exec_kind=1, reps=2)  # warm-up, first touch
        if reps is None:
            reps = int(max(min_reps, min(200, min_seconds / max(sec1, 1e-6))))
        _, sec = ref.spmv("csr", rp, ci, va, x, N_ROWS, exec_kind=1, reps=reps)
        kind = "reference"
    else:
        from oracle import oracle
        y = np.zeros(n)
        if reps is None:
            reps = max(1, min_reps // 4)
        t0 = time.perf_counter()
        for _ in range(reps):
            oracle.call("orc_csr_spmv_f64_i32", n, N_ROWS, nnz, rp, ci, va, x, 1, 1, y, 1)
        sec = (time.perf_counter() - t0) / reps
        cores, kind = 1, "port"
    return {"value": 2.0 * nnz / sec / 1e9, "unit": "GFLOP/s", "cores": cores, "kind": kind,
            "sample": "the full %s (n=%d, nnz=%d) against the full x; %s; %d reps, %.3f ms/SpMV; "
                      "OMP_PROC_BIND=%s OMP_PLACES=%s (set before libgomp loads), nproc=%d"
                      % (CFG, n, nnz, "gko::OmpExecutor Csr(classical)::apply, %d threads" % cores
                         if kind == "reference" else "oracle C port, 1 thread", reps, sec * 1e3,
                         os.environ.get("OMP_PROC_BIND"), os.environ.get("OMP_PLACES"), os.cpu_count() or 0),
            "ms": sec * 1e3, "nnz": nnz}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    b = cpu_reference_spmv(cfg2_on_host(), args.steps, reps=args.steps)
    line = {
        "impl": "reference", "metric": "csr_spmv_fp64_gflops", "value": b["value"],
        "unit": "GFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": b["ms"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: CSR SpMV fp64/int32, random n=%d nnz=%d (15 distinct uniform "
                               "cols/row), workloads.py seed 42" % (CFG, N_ROWS, N_ROWS * PER_ROW),
                   "cpu_arm": b["sample"]},
        "cpu_baseline": {k: b[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": b["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------ GPU arm
def run_gpu_arm(args, rank, world):
    import torch
    import torch.distributed as dist
    from ginkgo_b200 import api
    from ginkgo_b200 import distributed as D

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ex = api.HostExecutor(local)  # C++ host layer (gko_b200.hpp) over the C ABI
    dev = ex.device
    hl = api._host()
    dump = OutputDump(args.dump_outputs, world, ex.stream) if args.dump_outputs else None

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record(ex.stream)
        for _ in range(n):
            fn()
        e1.record(ex.stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---------------------------------------------------------------- SpMV, cfg2 (headline)
    offs = D.uniform_offsets(N_ROWS, world)
    r0, r1 = offs[rank], offs[rank + 1]
    with torch.cuda.stream(ex.stream):
        rp, ci, va = W.build(CFG, r0, r1, xp="torch", device=dev)
        x_full = W.vector(N_ROWS, xp="torch", device=dev)
    nnz_loc = va.numel()
    nnz_total = N_ROWS * PER_ROW
    if world == 1:
        A = api.host_csr(ex, (N_ROWS, N_ROWS), va, ci, rp)
        xg = api.host_dense(ex, x_full)
        y_t = torch.empty(N_ROWS, dtype=torch.float64, device=dev)
        yg = api.host_dense(ex, y_t)

        def step():
            api._hcheck(hl.gkob_apply(A.h, xg.h, yg.h))
        kernel_step = step
    else:
        def build_dist():
            A_ = api.DistMatrix(ex, offs, rp, ci, va)
            with torch.cuda.stream(ex.stream):
                xe = torch.zeros(A_.n_local + A_.n_ghost, dtype=torch.float64, device=dev)
                xe[:A_.n_local] = x_full[r0:r1]
                yt = torch.empty(A_.n_local, dtype=torch.float64, device=dev)
            Al = api.host_csr(ex, (A_.n_local, A_.n_local + A_.n_ghost), va, A_.col_idxs, rp)
            return A_, xe, yt, Al, api.host_dense(ex, xe), api.host_dense(ex, yt)

        def halo_delivers(A_, xe, yt):
            """one exchange: every ghost slot must hold the x entry of its global column (all ranks)"""
            A_.apply(xe, yt)
            ex.synchronize()
            with torch.cuda.stream(ex.stream):
                good = A_.n_ghost == 0 or torch.equal(A_.last_ghosts(), x_full[A_.part["ghosts"].to(dev).long()])
                t = torch.tensor([1 if good else 0], device=dev)
            ex.synchronize()
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return int(t.item()) == 1

        A, x_ext, y_t, Aloc, xe_h, y_h = build_dist()
        halo_path = "peer-memory halo exchange over NVLink" if A.p2p & 2 else "NCCL halo exchange"
        if not halo_delivers(A, x_ext, y_t):
            if not A.p2p:
                raise RuntimeError("the halo exchange delivers wrong ghost values")
            # same decision on every rank (all-reduced flag): rebuild on the NCCL path
            os.environ["B200_P2P"] = "0"
            del A, Aloc, xe_h, y_h
            A, x_ext, y_t, Aloc, xe_h, y_h = build_dist()
            halo_path = "NCCL halo exchange (the peer-memory exchange failed its validation on this box)"
            if not halo_delivers(A, x_ext, y_t):
                raise RuntimeError("the halo exchange delivers wrong ghost values")

        def step():  # halo exchange (referenced remote entries only) + local SpMV
            A.apply(x_ext, y_t)

        def kernel_step():
            api._hcheck(hl.gkob_apply(Aloc.h, xe_h.h, y_h.h))
    ex.synchronize()
    kernel_name = {2: "warp_stream_kernel", 4: "warp_pipe_kernel", 5: "ring_kernel"}.get(
        hl.gkob_csr_kernel_variant((A if world == 1 else Aloc).h), "warp_stream_kernel")
    plan_parts = hl.gkob_csr_plan_parts((A if world == 1 else Aloc).h)
    for _ in range(max(args.warmup, 3)):
        step()
    dist_modes = None
    with ClockSampler(local) as cs:
        l0 = ex.launch_count()
        ms_total = timed(step, args.steps)
        launches = ex.launch_count() - l0
        if dump:
            dump.take("csr_spmv_cfg2_y", y_t, r0, N_ROWS, 2 << 20)
        for _ in range(3):
            kernel_step()
        ms_kernel = timed(kernel_step, args.steps) / args.steps  # dominant kernel alone
        if world > 1:
            # second mode: exchange and SpMV pipelined by owner block (arrival-order row sums: must agree
            # with the exact mode to 1e-13, the SpMV tolerance of SURVEY.md section 8d)
            dist_modes = {"exact": {"ms_per_step": ms_total / args.steps,
                                    "exchange_ms_per_step": ms_total / args.steps - ms_kernel,
                                    "row_sums": "left to right, bit-identical to 1 GPU"}}
            with torch.cuda.stream(ex.stream):
                y_exact = y_t.clone()
            A.set_overlap(True)
            step()
            ex.synchronize()
            with torch.cuda.stream(ex.stream):
                pipe_on = bool(A.pipelined)
                pipe_diff = float(((y_t - y_exact).abs().max() / y_exact.abs().max()).item())
                dev_ok = pipe_on and pipe_diff <= 1e-13
                t = torch.tensor([1 if dev_ok else 0], device=dev)
            ex.synchronize()
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t.item()) == 1:
                for _ in range(3):
                    step()
                l0 = ex.launch_count()
                ms_ov = timed(step, args.steps)
                launches_ov = ex.launch_count() - l0
                dist_modes["pipelined"] = {"ms_per_step": ms_ov / args.steps,
                                           "row_sums": "owner blocks in arrival order, equal to the exact mode "
                                                       "to 1e-13 relative (checked in this run)"}
                if ms_ov < ms_total:
                    ms_total, launches = ms_ov, launches_ov
                    if dump:
                        dump.take("csr_spmv_cfg2_y", y_t, r0, N_ROWS, 2 << 20)
                    halo_path += "; exchange and SpMV pipelined by owner block (opt-in mode, 1e-13-equal row sums)"
                else:
                    A.set_overlap(False)
            else:
                A.set_overlap(False)
                dist_modes["pipelined"] = {"unavailable": "rank 0: pipelined apply ran = %s, max relative difference "
                                                          "to the exact mode = %.3e (gate 1e-13); not taken unless "
                                                          "every rank qualifies" % (pipe_on, pipe_diff)}
    ms_step = ms_total / args.steps
    value = 2.0 * nnz_total / (ms_step * 1e-3) / 1e9

    # ----------------------------- end to end with HOST buffers: H2D x, SpMV, D2H y
    n_e2e = max(5, min(args.steps, 50))
    if world == 1:
        # the public host-buffer call: gko_b200::staged_apply (Csr::apply with HOST b and x;
        # upload, kernel and download of consecutive calls overlap on three streams)
        xh = x_full.cpu().pin_memory()
        yh = torch.empty(N_ROWS, dtype=torch.float64).pin_memory()
        staged = api.StagedApply(A)

        def e2e_step():
            staged.apply(xh, yh)
        e2e_join = staged.join
        h2d, d2h = N_ROWS * 8, N_ROWS * 8
    else:
        xh = x_full[r0:r1].cpu().pin_memory()
        yh = torch.empty(A.n_local, dtype=torch.float64).pin_memory()

        def e2e_step():
            with torch.cuda.stream(ex.stream):
                x_ext[:A.n_local].copy_(xh, non_blocking=True)
            step()
            with torch.cuda.stream(ex.stream):
                yh.copy_(y_t, non_blocking=True)

        def e2e_join():
            pass
        h2d, d2h = N_ROWS * 8, N_ROWS * 8  # summed over ranks
    for _ in range(3):
        e2e_step()
    e2e_join()

    def e2e_run():  # n_e2e calls, then the compute stream waits for the last download
        for _ in range(n_e2e):
            e2e_step()
        e2e_join()
    ms_e2e = timed(e2e_run, 1) / n_e2e
    if world == 1:  # the pipelined result must be the SpMV result
        ex.synchronize()
        assert torch.equal(yh, y_t.cpu()), "staged apply disagrees with the device apply"
    e2e = {"value": 2.0 * nnz_total / (ms_e2e * 1e-3) / 1e9, "unit": "GFLOP/s",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e}

    peak, peak_src = peaks()
    ncols_loc = N_ROWS if world == 1 else A.n_local + A.n_ghost
    alg_bytes = W.spmv_bytes(r1 - r0, ncols_loc, nnz_loc)
    achieved = alg_bytes / (ms_kernel * 1e-3) / 1e9
    n_launch = max(plan_parts, 1)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "kernel": "b200::csr::%s<double,int,1,...>" % kernel_name + (
                    " x %d launches (column-blocked copy, parts applied in order)" % plan_parts
                    if plan_parts > 1 else ""),
                # one SpMV = `launches_per_step` launches of the kernel; bytes and time are per STEP
                "launches_per_step": n_launch,
                "algorithmic_bytes_per_step": alg_bytes, "kernel_ms_per_step": ms_kernel,
                "algorithmic_bytes_per_launch": alg_bytes / n_launch, "ms_per_launch": ms_kernel / n_launch,
                "gather_lines_per_element": hl.gkob_csr_gather_lines((A if world == 1 else Aloc).h)
                if hasattr(hl, "gkob_csr_gather_lines") else None}
    prof = os.path.join(ROOT, "profiles", "r02_csr_spmv_cfg2.json")
    if os.path.exists(prof) and world == 1:  # ncu --set full capture of THIS build's bench command
        try:
            pj = json.load(open(prof))
            if int(pj.get("launches_per_step", -1)) == n_launch:
                roofline["traffic"] = pj.get("dram_bytes_per_step")
                roofline["traffic_source"] = "profiles/r02_csr_spmv_cfg2.json (dram__bytes_read.sum + " \
                                             "dram__bytes_write.sum of the step's launches, ncu --set full)"
        except Exception:
            pass
    host_mat = None
    if world == 1 and not args.no_cpu:  # the CPU arm times the SAME matrix
        host_mat = tuple(t.cpu().numpy() for t in (rp, ci, va, x_full))
    del A, rp, ci, va
    torch.cuda.empty_cache()

    # ------------------------------------------ banded twin of cfg2 (same n, nnz/row; local gathers)
    twin = None
    if world == 1 and not args.no_twin:
        with torch.cuda.stream(ex.stream):
            brp, bci, bva = W.build("cfg2_banded", xp="torch", device=dev)
            yb = torch.empty(N_ROWS, dtype=torch.float64, device=dev)
        B = api.host_csr(ex, (N_ROWS, N_ROWS), bva, bci, brp)
        xb, ybh = api.host_dense(ex, x_full), api.host_dense(ex, yb)

        def bstep():
            api._hcheck(hl.gkob_apply(B.h, xb.h, ybh.h))
        for _ in range(3):
            bstep()
        ms_b = timed(bstep, args.steps) / args.steps
        if dump:
            dump.take("csr_spmv_cfg2_banded_y", yb, 0, N_ROWS, 1 << 20)
        bbytes = W.spmv_bytes(N_ROWS, N_ROWS, bva.numel())
        twin = {"workload": "banded twin of cfg2: n=%d, columns row-7..row+7, nnz=%d" % (N_ROWS, bva.numel()),
                "ms_per_step": ms_b, "gflops": 2.0 * bva.numel() / (ms_b * 1e-3) / 1e9,
                "achieved": bbytes / (ms_b * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": bbytes / (ms_b * 1e-3) / 1e9 / peak,
                "kernel_variant": hl.gkob_csr_kernel_variant(B.h)}
        del B, brp, bci, bva, yb
        torch.cuda.empty_cache()
    roofline["banded_twin"] = twin
    # ------------------------------------------ skewed twin: Zipf row lengths, the nnz of cfg2
    skew = None
    if world == 1 and not args.no_twin:
        with torch.cuda.stream(ex.stream):
            zrp, zci, zva = W.build("cfg2_zipf", xp="torch", device=dev)
            yz = torch.empty(N_ROWS, dtype=torch.float64, device=dev)
        Z = api.host_csr(ex, (N_ROWS, N_ROWS), zva, zci, zrp)
        xz, yzh = api.host_dense(ex, x_full), api.host_dense(ex, yz)

        def zstep():
            api._hcheck(hl.gkob_apply(Z.h, xz.h, yzh.h))
        for _ in range(3):
            zstep()
        ms_z = timed(zstep, args.steps) / args.steps
        if dump:
            dump.take("csr_spmv_cfg2_zipf_y", yz, 0, N_ROWS, 1 << 20)
        zbytes = W.spmv_bytes(N_ROWS, N_ROWS, zva.numel())
        with torch.cuda.stream(ex.stream):
            zl = (zrp[1:] - zrp[:-1])
            zmax, zlong = int(zl.max().item()), int((zl >= 1024).sum().item())
        skew = {"workload": "skewed twin of cfg2: n=%d, Zipf row lengths (longest row %d entries, %d rows >= 1024 "
                            "split over CTAs), nnz=%d, columns spread over all of x"
                            % (N_ROWS, zmax, zlong, zva.numel()),
                "ms_per_step": ms_z, "gflops": 2.0 * zva.numel() / (ms_z * 1e-3) / 1e9,
                "achieved": zbytes / (ms_z * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": zbytes / (ms_z * 1e-3) / 1e9 / peak, "kernel_variant": hl.gkob_csr_kernel_variant(Z.h),
                "vs_uniform_random_cfg2": (zbytes / ms_z) / (alg_bytes / ms_kernel)}
        del Z, zrp, zci, zva, yz
        torch.cuda.empty_cache()
    roofline["skewed_twin"] = skew
    del x_full

    # ------------------------------------------------------------------------------ CG
    cg = run_cg(args, rank, world, ex, dev, timed_events=True, dump=dump)

    if rank != 0:
        return
    if dump:
        dump.write()
    cpu = cpu_reference_spmv(host_mat, 10) if host_mat is not None else None
    line = {
        "metric": "csr_spmv_fp64_gflops", "value": value, "unit": "GFLOP/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "%s: CSR SpMV fp64/int32, random n=%d nnz=%d (15 distinct uniform "
                               "cols/row), workloads.py seed 42" % (CFG, N_ROWS, nnz_total),
                   "parallelism": "1-D row split over %d GPU(s)%s" %
                                  (world, ", %s of the referenced x entries per step" % halo_path
                                   if world > 1 else ""),
                   "dist_modes": dist_modes,
                   "l2": "inputs (2.0 GB/step) exceed the 126 MB L2; no flush between steps",
                   "gbs": alg_bytes * world / (ms_step * 1e-3) / 1e9},
        "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": cs.summary(),
        "cg": cg,
    }
    # the solver legs also under `config` (a key every consumer of the line keeps)
    line["config"]["solver_legs"] = {k: {kk: v[kk] for kk in ("iterations", "iters_per_s", "true_rel_residual",
                                                               "roofline") if kk in v}
                                     for k, v in cg.items()}
    if cpu:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))


def run_cg(args, rank, world, ex, dev, timed_events=True, dump=None):
    """CG iterations/s: N == 1 -> BASELINE configs[2] (7-pt Laplacian 200^3 + scalar Jacobi, to
    1e-8) AND configs[4] (400^3, 200 iterations); N > 1 -> configs[4] row-sharded (z-slabs)."""
    import torch
    import torch.distributed as dist
    from ginkgo_b200 import api
    from ginkgo_b200 import distributed as D
    out = {}

    def wall(fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ex.stream)
        fn()
        e1.record(ex.stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    if world == 1 and not args.no_cg:
        g = W.CONFIGS["cfg3"]["grid"]
        n = g ** 3
        with torch.cuda.stream(ex.stream):
            rp, ci, va = W.laplace(g, 3, xp="torch", device=dev)
            b = torch.ones(n, dtype=torch.float64, device=dev)
            x = torch.zeros(n, dtype=torch.float64, device=dev)
        A = api.host_csr(ex, (n, n), va, ci, rp)
        s = api.HostSolver(ex, "cg", A, precond_max_bs=1, max_iters=5000, reduction=1e-8, fused=True)
        bd, xd = api.host_dense(ex, b), api.host_dense(ex, x)
        s.apply(bd, xd)  # warm-up solve (builds the plan + graph)
        x.zero_()
        ms = wall(lambda: s.apply(bd, xd))
        if dump:
            dump.take("cg_cfg3_x", x, 0, n, 1 << 20)
        # true relative residual
        r = b.clone()
        rd = api.host_dense(ex, r)
        one = api.host_dense(ex, torch.ones(1, dtype=torch.float64, device=dev))
        neg = api.host_dense(ex, -torch.ones(1, dtype=torch.float64, device=dev))
        api._hcheck(api._host().gkob_apply4(A.h, neg.h, xd.h, one.h, rd.h))
        ex.synchronize()
        nnz = va.numel()
        bytes_it = nnz * 12 + (n + 1) * 4 + 13 * n * 8
        out["cfg3"] = {"workload": "cfg3: CG + scalar Jacobi fp64, 7-pt Laplacian 200^3, b=1, "
                                   "ResidualNorm(rhs_norm) 1e-8", "iterations": s.num_iterations,
                       "ms": ms, "iters_per_s": s.num_iterations / (ms * 1e-3),
                       "true_rel_residual": (r.norm() / b.norm()).item(),
                       "fused": s.used_fused, "stop_status": s.stop_status,
                       "algorithmic_gbs": bytes_it * s.num_iterations / (ms * 1e-3) / 1e9,
                       "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peaks()[0],
                                    "achieved": bytes_it * s.num_iterations / (ms * 1e-3) / 1e9,
                                    "frac": bytes_it * s.num_iterations / (ms * 1e-3) / 1e9 / peaks()[0],
                                    "bytes_model": "fused minimum per iteration: nnz*12 + (n+1)*4 + 13*n*8 "
                                                   "(SURVEY 8d; the reference's unfused count is +6*n*8)"}}
        del A, s, rp, ci, va, b, x, r
        torch.cuda.empty_cache()
    if args.no_cg:
        return out
    if world == 1 and not args.no_gmres:
        # configs[3]: GMRES(30, MGS) + block-Jacobi(16) fp32, random nonsymmetric diagonally
        # dominant n=4M nnz=80M, uniform block pointers, rel. residual 1e-6
        c4 = W.CONFIGS["cfg4"]
        n = c4["n"]
        with torch.cuda.stream(ex.stream):
            rp, ci, va = W.build("cfg4", xp="torch", device=dev)
            b = torch.ones(n, dtype=torch.float32, device=dev)
            x = torch.zeros(n, dtype=torch.float32, device=dev)
        A = api.host_csr(ex, (n, n), va, ci, rp)
        bp = np.arange(0, n + 1, 16, dtype=np.int32)
        t0 = time.perf_counter()
        s = api.HostSolver(ex, "gmres", A, precond_max_bs=16, block_ptrs=bp, max_iters=1000,
                           reduction=1e-6, krylov_dim=30, ortho=0)
        bd, xd = api.host_dense(ex, b), api.host_dense(ex, x)
        s.apply(bd, xd)  # warm-up (includes the host-side block inversion of the generate step)
        setup_s = time.perf_counter() - t0
        x.zero_()
        ms = wall(lambda: s.apply(bd, xd))
        if dump:
            dump.take("gmres_cfg4_x", x, 0, n, 1 << 20)
        r = b.clone()
        rd = api.host_dense(ex, r)
        one = api.host_dense(ex, torch.ones(1, dtype=torch.float32, device=dev))
        neg = api.host_dense(ex, -torch.ones(1, dtype=torch.float32, device=dev))
        api._hcheck(api._host().gkob_apply4(A.h, neg.h, xd.h, one.h, rd.h))
        ex.synchronize()
        out["cfg4"] = {"workload": "cfg4: GMRES(30, MGS) + block-Jacobi(16) fp32, random "
                                   "nonsymmetric diag-dominant n=4M nnz=80M, b=1, 1e-6",
                       "iterations": s.num_iterations, "ms": ms,
                       "iters_per_s": s.num_iterations / (ms * 1e-3),
                       "true_rel_residual": (r.double().norm() / b.double().norm()).item(),
                       "stop_status": s.stop_status, "first_apply_incl_generate_s": setup_s}
        # byte model of the reference (core/solver/gmres.cpp:427-443) with d = Krylov vectors actually
        # built before the stop: (5d/2 + 21/2 + 14/d) n V + (1 + 1/d) (B_matrix + B_blocks)
        d_ = max(1, min(30, s.num_iterations))
        nnz4 = va.numel()
        bmat = nnz4 * 8 + (n + 1) * 4
        bblk = (n // 16) * 256 * 4 + (n // 16 + 1) * 4
        bytes_it4 = (2.5 * d_ + 10.5 + 14.0 / d_) * n * 4 + (1 + 1.0 / d_) * (bmat + bblk)
        gbs4 = bytes_it4 * s.num_iterations / (ms * 1e-3) / 1e9
        out["cfg4"]["roofline"] = {"bound": "hbm", "unit": "GB/s", "peak": peaks()[0], "achieved": gbs4,
                                   "frac": gbs4 / peaks()[0],
                                   "bytes_model": "reference formula core/solver/gmres.cpp:427-443 with d=%d" % d_}
        del A, s, rp, ci, va, b, x, r
        torch.cuda.empty_cache()
    # configs[4]: 400^3, fixed 200 iterations (reduction 0 never triggers), strong scaling
    g = W.CONFIGS["cfg5"]["grid"] if not args.small_cg else 160
    n = g ** 3
    offs = [p * g // world * g * g for p in range(world + 1)]  # whole z-slabs per rank
    r0, r1 = offs[rank], offs[rank + 1]
    iters = 200
    with torch.cuda.stream(ex.stream):
        rp, ci, va = W.laplace(g, 3, r0, r1, xp="torch", device=dev)
        b = torch.ones(r1 - r0, dtype=torch.float64, device=dev)
        x = torch.zeros(r1 - r0, dtype=torch.float64, device=dev)
    nnz_loc = va.numel()
    if world == 1:
        A = api.host_csr(ex, (n, n), va, ci, rp)
        s = api.HostSolver(ex, "cg", A, max_iters=iters, reduction=1e-300, fused=True, check_every=int(os.environ.get("B200_BENCH_CHECK_EVERY", "20")))
        bd, xd = api.host_dense(ex, b), api.host_dense(ex, x)
        s.apply(bd, xd)
        x.zero_()
        ms = wall(lambda: s.apply(bd, xd))
        done, ghosts = s.num_iterations, 0
    else:
        def warm_up():
            """build + one untimed solve; every rank learns whether ALL ranks got through"""
            A_ = api.DistMatrix(ex, offs, rp, ci, va)
            A_.make_cg(scalar_jacobi=False, max_iters=iters, reduction=1e-300, check_every=int(os.environ.get("B200_BENCH_CHECK_EVERY", "20")))
            good, why = 1, ""
            try:
                good = 1 if A_.cg_apply(b, x)[0] > 0 else 0
            except Exception as e:  # noqa: BLE001 (a peer-memory wait that timed out)
                good, why = 0, repr(e)
            t = torch.tensor([good], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return A_, int(t.item()) == 1, why

        A, good, why = warm_up()
        if not good:
            if not A.p2p:
                raise RuntimeError("distributed CG failed: " + why)
            os.environ["B200_P2P"] = "0"  # same decision on every rank: NCCL collectives
            del A
            A, good, why = warm_up()
            if not good:
                raise RuntimeError("distributed CG failed: " + why)
        x.zero_()
        res = {}
        ms = wall(lambda: res.update(it=A.cg_apply(b, x)[0]))
        done, ghosts = res["it"], A.n_ghost
    if dump:
        dump.take("cg_cfg5_x", x, r0, n, 1 << 20)
    # TRUE residual ||b - A x|| / ||b|| of the timed solve, identical code path for every N
    # (a wrong halo inside the CG graph would show here); compared with the reference's
    # 200-iteration value (tests/golden/fullsize_reference.json) at the full size
    with torch.cuda.stream(ex.stream):
        yt = torch.empty(r1 - r0, dtype=torch.float64, device=dev)
        if world == 1:
            xe = x
        else:
            xe = torch.zeros(A.n_local + A.n_ghost, dtype=torch.float64, device=dev)
            xe[:A.n_local] = x
    if world == 1:
        xed, ytd = api.host_dense(ex, xe), api.host_dense(ex, yt)  # the handles must outlive the call
        api._hcheck(api._host().gkob_apply(A.h, xed.h, ytd.h))
    else:
        A.apply(xe, yt)
    ex.synchronize()
    with torch.cuda.stream(ex.stream):
        sq = torch.stack([((b - yt) ** 2).sum(), (b ** 2).sum()])
    ex.synchronize()
    if world > 1:
        dist.all_reduce(sq)
    true_res = float((sq[0] / sq[1]).sqrt().item())
    ref_res = None
    try:
        gj = json.load(open(os.path.join(ROOT, "tests", "golden", "fullsize_reference.json")))
        if not args.small_cg and "cfg5" in gj:
            ref_res = gj["cfg5"]["true_rel_residual"]
    except Exception:
        pass
    if ref_res is not None and done == iters and abs(true_res - ref_res) > 1e-10 + 1e-6 * ref_res:
        raise RuntimeError("cfg5 CG on %d GPU(s): true residual %.12e after %d iterations, the reference "
                           "has %.12e" % (world, true_res, done, ref_res))
    nnz_t = torch.tensor([nnz_loc], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(nnz_t)
    nnz = int(nnz_t.item())
    bytes_it = nnz * 12 + (n + world) * 4 + 13 * n * 8
    peak, _ = peaks()
    gbs = bytes_it * done / (ms * 1e-3) / 1e9
    out["cfg5"] = {"workload": "cfg5: CG fp64 (unpreconditioned), 7-pt Laplacian %d^3 n=%d nnz=%d, "
                               "b=1, %d iterations, rows split in z-slabs over %d GPU(s)"
                               % (g, n, nnz, iters, world), "iterations": done, "ms": ms,
                   "iters_per_s": done / (ms * 1e-3), "ghosts_per_rank": ghosts,
                   "collectives": ("single GPU" if world == 1 else
                                   "peer memory over NVLink" if A.p2p else "NCCL"),
                   "true_rel_residual": true_res, "reference_true_rel_residual": ref_res,
                   "algorithmic_gbs": gbs,
                   "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak * world, "unit": "GB/s",
                                "frac": gbs / (peak * world),
                                "bytes_model": "fused minimum per iteration: nnz*12 + (n+1)*4 + 13*n*8 (SURVEY 8d)"}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cg", action="store_true", help="skip the CG legs")
    ap.add_argument("--no-gmres", action="store_true", help="skip the GMRES + block-Jacobi leg")
    ap.add_argument("--no-twin", action="store_true", help="skip the banded twin of cfg2")
    ap.add_argument("--small-cg", action="store_true", help="160^3 instead of 400^3 for the cfg5 leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of every timed leg's result to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU legs; --impl reference has none")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    run_gpu_arm(args, rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
