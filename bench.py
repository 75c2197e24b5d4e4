#!/usr/bin/env python
"""bench.py -- headline benchmark of the LIBXSMM hot path on B200 (contract: one JSON line on stdout).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload brgemm|fsspmdm|bcsc|sweep]
                  [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): batched BRGEMM bf16 x bf16 -> f32, m=n=k=64, br=8 (stride mode),
batch = 65536 independent tiles PER GPU with all operands unique ("mode S" of SURVEY.md 8d). One step is
one pass over the batch = ONE launch of the tcgen05 tile kernel through the C ABI
(libxsmm_b200_gemm_batch_strided). Inputs (8.6 GB) are far larger than L2, so no flush is needed.

  value  whole-job GFLOP/s, operands resident in HBM, CUDA events on the launching stream, max over ranks
  e2e    same metric through the same C-ABI call with HOST (pinned) buffers: H2D + kernel + D2H per step
  roofline      achieved algorithmic GB/s of the dominant kernel vs the measured HBM peak
  cpu_baseline  the reference's own JIT kernel (oracle/_ref, all host cores) on a bounded sample
  also          fsspmdm (config 3) and BCSC (config 4) with their own roofline numbers

--dump-outputs DIR writes the output of the timed path's last step as DIR/<name>.npy (float32), a fixed seeded sample of
DUMP_CHUNK-element chunks where it is larger than DUMP_BYTES; the inputs are seeded, so two builds can be compared output
for output.

--impl reference runs the unmodified reference (AMX/AVX-512 JIT through its public dispatch API, OpenMP over
the batch) on a bounded sample of the same workload on rank 0 only.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

M = N = K = 64
BR = 8
BATCH = 65536
BF16, F32 = 2, 1
FLAG_BETA_0 = 4
METRIC = "batched BRGEMM GFLOP/s (bf16, m=n=k=64, br=8, batch=65536/GPU, unique operands)"
WORKLOAD = ("configs[1]: batched BRGEMM bf16->f32 m=n=k=64 brcount=8 batch=65536 per GPU, stride-BR, beta=0, "
            "mode S (all operands unique)")
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed `ncu --set full` captures (bytes)
NCU_TRAFFIC = {"gemm_tc_kernel<64>": (9673.1e6, "profiles/r02_ncu_gemm_tc.txt"),
               "sreg_kernel<float>": (622.1e6, "profiles/r02_ncu_sreg.txt"),
               "bcsc_ts_kernel<32,2>": (491.3e6, "profiles/r02_ncu_bcsc_ts.txt"),       # below the 537 MB of algorithmic bytes: part of C is still in L2 when the capture ends
               "gemm_pool_kernel": (495.2e6, "profiles/r02_ncu_gemm_pool.txt"),           # C writes (537 MB algorithmic); the operand pools stay in L2
               "gemm_ts_kernel": (745.9e6, "profiles/r02_ncu_gemm_ts_i8.txt")}


def traffic(kernel):
    t = NCU_TRAFFIC.get(kernel, (None, None))
    return t[0]


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "src": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        p = {"hbm_gbs": float(j["hbm_gbs"]), "bf16_tflops": float(j["bf16_tflops"]), "src": "measured"}
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.stop_flag, self.index = [], False, index
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.thread.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def fill_tenths(t, torch, chunk=1 << 26):
    """multiples of 0.1 in [-0.5, 0.5] like the reference drivers (spmm_kernel.c:498-527), seed 555"""
    g = torch.Generator(device=t.device); g.manual_seed(555)
    flat = t.view(-1)
    for s in range(0, flat.numel(), chunk):
        e = min(flat.numel(), s + chunk)
        flat[s:e] = (torch.randint(-5, 6, (e - s,), device=t.device, generator=g, dtype=torch.int8).to(torch.float32) / 10).to(t.dtype)


DUMP_BYTES = 16 << 20        # per output; at most four outputs are written, 64 MB in all
DUMP_CHUNK = 4096


def dump_outputs(args, torch, **outs):
    """the outputs of the timed path (device tensors) as float32 .npy files under args.dump_outputs"""
    if not args.dump_outputs or int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    assert len(outs) <= 4
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, t in outs.items():
        flat = t.reshape(-1)
        chunks = flat.numel() // DUMP_CHUNK
        keep = DUMP_BYTES // 4 // DUMP_CHUNK
        if chunks > keep:
            idx = np.sort(np.random.default_rng(555).choice(chunks, keep, replace=False))
            flat = flat[:chunks * DUMP_CHUNK].view(chunks, DUMP_CHUNK)[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(args.dump_outputs, name + ".npy"), flat.float().cpu().numpy().ravel())


def time_steps(torch, fn, steps, warmup, dist=None):
    """W warm-up + K timed steps between barrier+synchronize; CUDA events on the launching stream; max over ranks"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
        torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
        torch.cuda.synchronize()
    per = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    total_ms = ev[0].elapsed_time(ev[steps])
    if dist is not None:
        t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    return total_ms, per


# ------------------------------------------------------------------------------------------------ BRGEMM
def brgemm_setup(X, torch, batch, out_f32=True):
    tc = F32 if out_f32 else BF16
    shape = X.libxsmm_create_gemm_shape(M, N, K, M, K, M, BF16, BF16, tc, F32)
    cfg = X.libxsmm_create_gemm_batch_reduce_config(X.GEMM_BATCH_REDUCE_STRIDE, M * K * 2, K * N * 2, 0)
    kernel = X.libxsmm_dispatch_brgemm(shape, FLAG_BETA_0, 0, cfg)
    assert kernel, "dispatch failed"
    assert X.libxsmm_b200_kernel_backend(kernel) == X.BACKEND_TCGEN05, "tcgen05 kernel not selected"
    a = torch.empty(batch * BR * M * K, dtype=torch.bfloat16, device="cuda")
    b = torch.empty(batch * BR * K * N, dtype=torch.bfloat16, device="cuda")
    c = torch.empty(batch * M * N, dtype=torch.float32 if out_f32 else torch.bfloat16, device="cuda")
    fill_tenths(a, torch); fill_tenths(b, torch)
    strides = (BR * M * K * 2, BR * K * N * 2, M * N * (4 if out_f32 else 2))
    return kernel, a, b, c, strides


def brgemm_check(X, torch, a, b, c, strides, ntiles=4):
    """a few tiles against the CPU oracle (test infrastructure used as the checker only)"""
    import numpy as np
    from oracle_ffi import oracle, run_gemm
    import gen
    for t in (0, 1, 77, BATCH // 3)[:ntiles]:
        if (t + 1) * M * N > c.numel():
            continue
        ah = a[t * BR * M * K:(t + 1) * BR * M * K].view(torch.int16).cpu().numpy().view(np.uint16)
        bh = b[t * BR * K * N:(t + 1) * BR * K * N].view(torch.int16).cpu().numpy().view(np.uint16)
        want = np.zeros(M * N, dtype=np.float32)
        assert run_gemm(oracle, (M, N, K, M, K, M), (BF16, BF16, F32, F32), FLAG_BETA_0, 3, M * K * 2, K * N * 2, BR, ah, bh, want) == 0
        got = c[t * M * N:(t + 1) * M * N].float().cpu().numpy()
        err = gen.normf_rel(want, got)
        assert err < 1.2e-5, "bench output differs from the oracle (tile %d, err %g)" % (t, err)


def run_ours(args):
    import torch
    import libxsmm_b200 as X
    dist = None
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    X.libxsmm_b200_set_device(local)
    X.libxsmm_b200_set_stream(torch.cuda.current_stream().cuda_stream)
    X.libxsmm_b200_set_blocking(0)
    pk = peaks()
    out = {}
    if args.workload == "brgemm":
        kernel, a, b, c, (sa, sb, sc) = brgemm_setup(X, torch, BATCH)

        def step():
            rc = X.libxsmm_b200_gemm_batch_strided(kernel, a.data_ptr(), b.data_ptr(), c.data_ptr(), sa, sb, sc, BR, BATCH)
            assert rc == 0, X.libxsmm_b200_last_error_string()
        launches0 = X.libxsmm_b200_launch_count()
        step(); X.check(); brgemm_check(X, torch, a, b, c, (sa, sb, sc))
        launches0 = X.libxsmm_b200_launch_count()
        with ClockSampler(local) as clocks:
            total_ms, per = time_steps(torch, step, args.steps, args.warmup, dist)
        launches = X.libxsmm_b200_launch_count() - launches0 - args.warmup
        X.check()
        dump_outputs(args, torch, c=c)
        from libxsmm_b200.shard import weak_batch
        per_gpu, job_tiles = weak_batch(BATCH, world)      # batch is the only shard axis: every rank owns BATCH tiles, no collective
        flops = 2.0 * M * N * K * BR * per_gpu
        bytes_alg = float(BATCH) * (sa + sb + sc)
        ms = total_ms / args.steps
        kern_ms = sorted(per)[len(per) // 2]
        value = (2.0 * M * N * K * BR * job_tiles) / (ms * 1e-3) / 1e9     # whole job; ms is the max over ranks
        ach = bytes_alg / (kern_ms * 1e-3) / 1e9
        out = {"metric": METRIC, "value": value, "unit": "GFLOP/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": WORKLOAD,
                          "batch_per_gpu": BATCH, "parallelism": "batch sharded, no collective", "l2_policy": "inputs (8.6 GB) larger than L2, no flush"},
               "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": traffic("gemm_tc_kernel<64>"),
                            "traffic_src": NCU_TRAFFIC["gemm_tc_kernel<64>"][1], "algorithmic_bytes": bytes_alg,
                            "peak_src": pk["src"], "kernel": "gemm_tc_kernel<64>", "kernel_ms": kern_ms,
                            "tensor_frac_of_measured_bf16_peak": (flops / (kern_ms * 1e-3) / 1e12) / pk["bf16_tflops"]},
               "gpu_launches": int(launches), "clocks": clocks.summary()}
        if not args.no_e2e:
            # every rank drives its own GPU over its own PCIe link at the same time; whole-job value = all tiles / slowest rank
            try:
                old_aff = os.sched_getaffinity(0)
            except Exception:
                old_aff = None
            bind_to_gpu_numa_node(torch, local)
            out["e2e"] = brgemm_e2e(X, torch, kernel, a, b, sa, sb, sc, flops, c_dev=c, dist=dist, world=world)
            if old_aff:
                os.sched_setaffinity(0, old_aff)        # the CPU baselines below use every core again
        if world > 1 and not args.no_also:
            out["strong"] = strong_scaling(X, torch, pk, args, dist, world, rank)
        if rank == 0 and not args.no_also:
            out["also"] = {}
            for name, fn in (("fsspmdm", also_fsspmdm), ("bcsc", also_bcsc), ("brgemm_r", also_brgemm_r), ("sweep", sweep), ("meltw", also_meltw)):
                try:
                    out["also"][name] = fn(X, torch, pk, args)
                except Exception as e:  # secondary numbers must not take the headline down
                    out["also"][name] = {"error": repr(e)[:200]}
        if rank == 0 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline_brgemm()
    elif args.workload == "fsspmdm":
        out = also_fsspmdm(X, torch, pk, args, full=True)
    elif args.workload == "bcsc":
        out = also_bcsc(X, torch, pk, args, full=True)
    elif args.workload == "brgemm_r":
        out = also_brgemm_r(X, torch, pk, args, full=True)
    elif args.workload == "sweep":
        out = sweep(X, torch, pk, args, full=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def bind_to_gpu_numa_node(torch, local):
    """run this rank's host side (pinned allocations are first-touched here) on the CPUs next to its GPU"""
    try:
        pr = torch.cuda.get_device_properties(local)
        dev = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % dev) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def brgemm_e2e(X, torch, kernel, a, b, sa, sb, sc, flops, steps=3, c_dev=None, dist=None, world=1):
    """same call, HOST pinned buffers: the library moves A and B to the device, runs the kernel and brings C back inside the
    step. Two transports are timed: the chunked three-stream copy pipeline (default) and in-place access to the pinned
    buffers from the kernel (LIBXSMM_B200_ZEROCOPY=1); the better one is the e2e value, both are reported. With N ranks every
    rank runs the call on its own GPU at the same time (barrier before each step); a step costs the slowest rank's time."""
    nb_a, nb_b, nb_c = BATCH * sa, BATCH * sb, BATCH * sc
    ha = torch.empty(nb_a // 2, dtype=torch.bfloat16, pin_memory=True); hb = torch.empty(nb_b // 2, dtype=torch.bfloat16, pin_memory=True)
    hc = torch.empty(nb_c // 4, dtype=torch.float32, pin_memory=True)
    ha.copy_(a); hb.copy_(b)          # the synthetic operands, now resident on the host
    X.libxsmm_b200_set_blocking(1)
    res = {}
    for mode, env in (("copy_pipeline", None), ("zero_copy", "1")):
        if env is None:
            os.environ.pop("LIBXSMM_B200_ZEROCOPY", None)
        else:
            os.environ["LIBXSMM_B200_ZEROCOPY"] = env
        best = None
        for i in range(steps + 1):
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            rc = X.libxsmm_b200_gemm_batch_strided(kernel, ha.data_ptr(), hb.data_ptr(), hc.data_ptr(), sa, sb, sc, BR, BATCH)
            torch.cuda.synchronize(); dt = time.perf_counter() - t0
            assert rc == 0, X.libxsmm_b200_last_error_string()
            if dist is not None:
                t = torch.tensor([dt], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            if i > 0:
                best = dt if best is None else min(best, dt)
        res[mode] = best
        if c_dev is not None:      # the host result of this transport equals the device-resident run (same kernel, same inputs)
            n = 1 << 20
            assert torch.equal(hc[:n], c_dev[:n].cpu()) and torch.equal(hc[-n:], c_dev[-n:].cpu()), "e2e result differs (%s)" % mode
    os.environ.pop("LIBXSMM_B200_ZEROCOPY", None)
    X.libxsmm_b200_set_blocking(0)
    mode = min(res, key=res.get)
    best = res[mode]
    return {"value": world * flops / best / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": int(world * (nb_a + nb_b)), "d2h_bytes_per_step": int(world * nb_c),
            "ms_per_step": best * 1e3, "transport": mode, "ms_by_transport": {k: v * 1e3 for k, v in res.items()}, "ranks": world,
            "pcie_gbs_per_gpu": (nb_a + nb_b + nb_c) / best / 1e9,
            "note": "every rank at once: pinned host A,B -> libxsmm_b200_gemm_batch_strided -> pinned host C on its own GPU; wall clock around the "
                    "blocking call, max over ranks, best of %d; bytes are the whole job's" % steps}


def also_fsspmdm(X, torch, pk, args, full=False, n_cols=1000000, dist=None):
    import numpy as np
    Mf, Kf, Nf = 32, 128, n_cols
    rng = np.random.default_rng(555)
    a = ((rng.integers(-5, 6, size=Mf * Kf) / 10.0) * (rng.random(Mf * Kf) < 0.15)).astype(np.float32)
    nnz = int(np.count_nonzero(a))
    one = np.array([1.0], dtype=np.float32); zero = np.array([0.0], dtype=np.float32)
    h = X.libxsmm_fsspmdm_create(F32, Mf, Nf, Kf, Kf, Nf, Nf, one.ctypes.data, zero.ctypes.data, a.ctypes.data, 0, None)
    assert h
    g = torch.Generator(device="cuda"); g.manual_seed(555)
    b = torch.randn(Kf * Nf, device="cuda", generator=g); c = torch.empty(Mf * Nf, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step():
        X.libxsmm_fsspmdm_execute(h, b.data_ptr(), c.data_ptr())
    step(); X.check()
    checked = fsspmdm_check(torch, a, b, c, Mf, Kf, Nf)
    steps = args.steps if full else max(5, args.steps)
    total_ms, per = time_steps(torch, step, steps, 3, dist)
    X.check()
    if full:
        dump_outputs(args, torch, c=c)
    ms = sorted(per)[len(per) // 2] if dist is None else total_ms / steps
    bytes_alg = 4.0 * (Kf * Nf + Mf * Nf)
    ach = bytes_alg / (ms * 1e-3) / 1e9
    X.libxsmm_fsspmdm_destroy(h)
    cpu = None
    if dist is None and (full or not getattr(args, "no_cpu", False)):
        cpu = cpu_baseline_fsspmdm(a, Mf, Kf, nnz)
    return {"cpu_baseline": cpu, "metric": "fsspmdm GFLOP/s (f32 M=32 K=128 N=1e6, 15% nnz)", "value": 2.0 * nnz * Nf / (ms * 1e-3) / 1e9, "unit": "GFLOP/s (sparse)",
            "dense_equiv_gflops": 2.0 * Mf * Kf * Nf / (ms * 1e-3) / 1e9, "ms_per_step": ms, "nnz": nnz, "oracle_check": checked,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": traffic("sreg_kernel<float>"), "algorithmic_bytes": bytes_alg, "kernel": "sreg_kernel<float>"},
            "config": {"workload": "configs[2]: fsspmdm f32 M=32 K=128 N=1e6 15% nnz beta=0; B+C = 640 MB per step (> L2)"}}


def fsspmdm_check(torch, a_dense, b, c, Mf, Kf, Nf, width=256):
    """three column strips of the timed output (first, middle, last) against the CPU oracle (checker only)"""
    import numpy as np
    from oracle_ffi import oracle
    import gen
    one = np.array([1.0], dtype=np.float32); zero = np.array([0.0], dtype=np.float32)
    worst = 0.0
    starts = (0, (Nf // 2) // 16 * 16, Nf - width)
    for n0 in starts:
        bs = b.view(Kf, Nf)[:, n0:n0 + width].contiguous().cpu().numpy().ravel()
        want = np.zeros(Mf * width, dtype=np.float32)
        assert oracle["fsspmdm"](F32, Mf, width, Kf, Kf, width, width, one.ctypes.data, zero.ctypes.data, a_dense.ctypes.data, bs.ctypes.data, want.ctypes.data) == 0
        got = c.view(Mf, Nf)[:, n0:n0 + width].contiguous().cpu().numpy().ravel()
        err = gen.normf_rel(want, got)
        assert err < 1e-4, "fsspmdm bench output differs from the oracle (columns %d.., err %g)" % (n0, err)
        worst = max(worst, err)
    return {"strips": len(starts), "width": width, "max_normf_rel": worst}


def bcsc_check(torch, a, bv, c, colptr, rowidx, geo, mblocks, picks=None):
    """a few m_blocks of the timed output against the CPU oracle (driver gold spmm_kernel.c:74-217 restated)"""
    import numpy as np
    from oracle_ffi import oracle, iarr
    import gen
    Mb, Kb, Nb, bk, bn = geo
    bvh = bv.view(torch.int16).cpu().numpy().view(np.uint16)
    worst = 0.0
    picks = picks or sorted({0, 1, mblocks // 2 + 1, mblocks - 1})
    for mb in picks:
        ah = a[mb * Kb * Mb:(mb + 1) * Kb * Mb].view(torch.int16).cpu().numpy().view(np.uint16)
        want = np.zeros(Nb * Mb, dtype=np.uint16)
        assert oracle["bcsc"](iarr(BF16, BF16, F32, BF16), iarr(1, Mb, Kb, Nb, bk, bn), FLAG_BETA_0 | 256, ah.ctypes.data, bvh.ctypes.data,
                              colptr.ctypes.data, rowidx.ctypes.data, want.ctypes.data) == 0
        got = c[mb * Nb * Mb:(mb + 1) * Nb * Mb].view(torch.int16).cpu().numpy().view(np.uint16)
        err = gen.normf_rel(gen.to_f64(want, BF16), gen.to_f64(got, BF16))
        assert err <= 5e-3, "BCSC bench output differs from the oracle (m_block %d, err %g)" % (mb, err)   # bf16 threshold of spmm_kernel.c:1019-1029
        worst = max(worst, err)
    return {"m_blocks": len(picks), "max_normf_rel": worst}


def also_bcsc(X, torch, pk, args, full=False, mblocks=8192, dist=None):
    import numpy as np
    Mb, Kb, Nb, bk, bn = 32, 512, 512, 32, 32
    rng = np.random.default_rng(555)
    nbr, nbc = Kb // bk, Nb // bn
    keep = np.zeros(nbr * nbc, dtype=bool); keep[rng.permutation(nbr * nbc)[:nbr * nbc // 2]] = True
    keep = keep.reshape(nbc, nbr)
    colptr = np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.uint32); rowidx = np.nonzero(keep)[1].astype(np.uint32)
    nnzb = int(colptr[-1])
    shape = X.libxsmm_create_gemm_shape(mblocks, 0, Kb, Kb, 0, Nb, BF16, BF16, BF16, F32)
    kernel = X.libxsmm_create_packed_spgemm_bcsc(shape, FLAG_BETA_0 | X.GEMM_FLAG_VNNI_A, 0, X.SpgemmConfig(Mb, bk, bn))
    assert kernel
    a = torch.empty(mblocks * Kb * Mb, dtype=torch.bfloat16, device="cuda"); fill_tenths(a, torch)
    bv = torch.empty(nnzb * bk * bn, dtype=torch.bfloat16, device="cuda"); fill_tenths(bv, torch)
    c = torch.empty(mblocks * Nb * Mb, dtype=torch.bfloat16, device="cuda")
    d_cp = torch.from_numpy(colptr.view(np.int32).copy()).cuda(); d_ri = torch.from_numpy(rowidx.view(np.int32).copy()).cuda()
    p = X.GemmParam(); nb = C.c_ulonglong(nbc)
    p.a.primary, p.b.primary, p.b.secondary, p.b.tertiary, p.b.quaternary, p.c.primary = a.data_ptr(), bv.data_ptr(), d_cp.data_ptr(), d_ri.data_ptr(), C.addressof(nb), c.data_ptr()
    fn = X.GEMMFUNCTION(kernel)

    def step():
        fn(C.byref(p))
    step(); X.check()
    checked = bcsc_check(torch, a, bv, c, colptr, rowidx, (Mb, Kb, Nb, bk, bn), mblocks)
    variant = int(X.libxsmm_b200_bcsc_variant(kernel, nbc))
    assert variant in (1, 2), "BCSC bench did not take a tcgen05 kernel (variant %d)" % variant
    kname = "bcsc_ts_kernel<32,2>" if variant == 2 else "bcsc_tc_kernel<32>"
    steps = args.steps if full else max(3, args.steps // 4)
    total_ms, per = time_steps(torch, step, steps, 3, dist)
    X.check()
    if full:
        dump_outputs(args, torch, c=c)
    ms = sorted(per)[len(per) // 2] if dist is None else total_ms / steps
    bytes_alg = 2.0 * (mblocks * Kb * Mb + mblocks * Nb * Mb) + 2.0 * nnzb * bk * bn
    ach = bytes_alg / (ms * 1e-3) / 1e9
    X.libxsmm_release_kernel(kernel)
    cpu = None
    if dist is None and mblocks == 8192 and (full or not getattr(args, "no_cpu", False)):
        cpu = cpu_baseline_bcsc(colptr, rowidx, nnzb, (Mb, Kb, Nb, bk, bn))
    return {"cpu_baseline": cpu, "metric": "BCSC spmm GFLOP/s dense-equivalent (bf16, M=32 N=K=512, 32x32 blocks, 50%, m_blocks=8192)",
            "value": 2.0 * Mb * mblocks * Nb * Kb / (ms * 1e-3) / 1e9, "unit": "GFLOP/s (dense-equivalent)",
            "effective_gflops": 2.0 * Mb * mblocks * nnzb * bk * bn / (ms * 1e-3) / 1e9, "ms_per_step": ms, "oracle_check": checked,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": traffic(kname), "algorithmic_bytes": bytes_alg,
                         "kernel": kname + " (+ bcsc_prep_kernel, bcsc_pack_b_kernel: the timed call is all three launches)"},
            "config": {"workload": "configs[3] on one GPU: BCSC bf16 M=32 N=K=512 bk=bn=32 50% m_blocks=8192; A+C = 537 MB per step (> L2)"}}


def sweep_check(torch, a, b, c, m, types, flags, esz, csz, batch):
    """first, middle and last tile of a sweep point against the CPU oracle: integers bit-exact, f16 within 1e-3 (normf_rel)"""
    import numpy as np
    from oracle_ffi import oracle, run_gemm
    import gen
    worst = 0.0
    a8, b8, c8 = a.view(torch.uint8), b.view(torch.uint8), c.view(torch.uint8)
    for t in (0, batch // 2, batch - 1):
        ah = a8[t * m * m * esz:(t + 1) * m * m * esz].cpu().numpy(); bh = b8[t * m * m * esz:(t + 1) * m * m * esz].cpu().numpy()
        got = c8[t * m * m * csz:(t + 1) * m * m * csz].cpu().numpy()
        want = np.zeros(m * m * csz, dtype=np.uint8)
        assert run_gemm(oracle, (m, m, m, m, m, m), types, flags, 0, 0, 0, 1, ah, bh, want) == 0
        if esz == 1:
            assert np.array_equal(got, want), "sweep int8 m=%d tile %d differs from the oracle" % (m, t)
        else:
            err = gen.normf_rel(want.view(np.float32), got.view(np.float32))
            assert err < 1e-3, "sweep f16 m=%d tile %d differs from the oracle (err %g)" % (m, t, err)
            worst = max(worst, err)
    return {"tiles": 3, "max_normf_rel": worst, "bit_exact": esz == 1}


def sweep(X, torch, pk, args, batch=32768, full=False):
    """configs[4]: int8 x int8 -> int32 (U8 x I8, VNNI4 A) and F16 x F16 -> F32, m=n=k in {8..128}, br=1, unique operands"""
    I8, U8, I32, F16 = 12, 13, 8, 3
    pts, outs = [], {}
    for name, ta, tb, tcc, tcomp, flags, esz, csz in (("u8*i8->i32", U8, I8, I32, I32, FLAG_BETA_0 | X.GEMM_FLAG_VNNI_A, 1, 4),
                                                       ("f16*f16->f32", F16, F16, F32, F32, FLAG_BETA_0, 2, 4)):
        for m in (8, 16, 32, 64, 128):
            shape = X.libxsmm_create_gemm_shape(m, m, m, m, m, m, ta, tb, tcc, tcomp)
            kernel = X.libxsmm_dispatch_gemm(shape, flags, 0)
            if not kernel:
                pts.append({"type": name, "m": m, "error": "dispatch returned NULL"}); continue
            g = torch.Generator(device="cuda"); g.manual_seed(555 + m)
            a = torch.randint(0, 5, (batch * m * m * esz,), dtype=torch.uint8, device="cuda", generator=g)
            b = torch.randint(0, 5, (batch * m * m * esz,), dtype=torch.uint8, device="cuda", generator=g)
            if esz == 2:
                a = (torch.randint(-5, 6, (batch * m * m,), device="cuda", generator=g).float() / 10).half(); b = a.roll(7)
            c = torch.empty(batch * m * m * csz, dtype=torch.uint8, device="cuda")
            sa = sb = m * m * esz; sc = m * m * csz

            def step():
                rc = X.libxsmm_b200_gemm_batch_strided(kernel, a.data_ptr(), b.data_ptr(), c.data_ptr(), sa, sb, sc, 1, batch)
                assert rc == 0, X.libxsmm_b200_last_error_string()
            step(); X.check()
            chk = sweep_check(torch, a, b, c, m, (ta, tb, tcomp, tcc), flags, esz, csz, batch)
            total_ms, per = time_steps(torch, step, args.steps if full else max(5, args.steps // 2), 3)
            X.check()
            if full and m == 128:
                outs[name.split("->")[0].replace("*", "_")] = c.view(torch.int32 if esz == 1 else torch.float32)
            ms = sorted(per)[len(per) // 2]
            bytes_alg = float(batch) * (sa + sb + sc)
            ach = bytes_alg / (ms * 1e-3) / 1e9
            pts.append({"type": name, "m": m, "gflops": 2.0 * m * m * m * batch / (ms * 1e-3) / 1e9, "ms": ms, "gbs": ach, "hbm_frac": ach / pk["hbm_gbs"],
                        "backend": int(X.libxsmm_b200_kernel_backend(kernel)), "oracle_check": chk, "l2_note": "operands %.0f MB%s" % (bytes_alg / 1e6, "" if bytes_alg > 2.5e8 else " (fits L2: not an HBM number)")})
    dump_outputs(args, torch, **outs)
    best = max((p for p in pts if "gflops" in p), key=lambda p: p["gflops"])
    return {"metric": "mixed-precision sweep GFLOP/s (configs[4], diagonal m=n=k)", "value": best["gflops"], "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps,
            "warmup": 3, "higher_is_better": True, "dtype": "u8/i8->i32, f16->f32", "data": "synthetic",
            "config": {"workload": "configs[4]: int8 and f16 GEMM m=n=k in {8,16,32,64,128}, batch=32768, br=1, beta=0, unique operands"},
            "points": pts, "roofline": {"bound": "hbm", "achieved": best["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": best["hbm_frac"], "traffic": None}}


def also_brgemm_r(X, torch, pk, args, full=False, pool_sets=64, batch=BATCH):
    """SURVEY.md 8d "mode R": the same 64^3 x 8 bf16 BRGEMM, ADDRESS batch-reduce, every tile's A block-set and B block-set drawn
    from a pool of 64 sets each (8 MB, L2-resident), C unique bf16 -- the tensor-core-bound variant of configs[1]. One step = one
    libxsmm_b200_gemm_plan_run over 65536 per-tile argument structs (the plan sorts tiles by set pair; equal neighbours share their
    operands in shared memory; pairs of tiles with the same B set share one M=128 instruction). Roofline: dense bf16 tensor throughput
    (MEASURED_PEAKS bf16_tflops, burst: the kernel is timed alone)."""
    import numpy as np
    from oracle_ffi import oracle, run_gemm
    import gen
    shape = X.libxsmm_create_gemm_shape(M, N, K, M, K, M, BF16, BF16, BF16, F32)
    cfg = X.libxsmm_create_gemm_batch_reduce_config(X.GEMM_BATCH_REDUCE_ADDRESS, 0, 0, 0)
    kernel = X.libxsmm_dispatch_brgemm(shape, FLAG_BETA_0, 0, cfg)
    assert kernel
    blk = M * K * 2
    pool_a = torch.empty(pool_sets * BR * M * K, dtype=torch.bfloat16, device="cuda"); fill_tenths(pool_a, torch)
    pool_b = torch.empty(pool_sets * BR * K * N, dtype=torch.bfloat16, device="cuda"); fill_tenths(pool_b, torch); pool_b = pool_b.roll(977)
    c = torch.empty(batch * M * N, dtype=torch.bfloat16, device="cuda")
    rng = np.random.default_rng(555)
    sa = rng.integers(0, pool_sets, size=batch); sb = rng.integers(0, pool_sets, size=batch)
    # per-tile argument structs exactly as a reference caller fills them (pointer arrays of br blocks)
    pa = (pool_a.data_ptr() + (sa[:, None] * BR + np.arange(BR)[None, :]) * blk).astype(np.uint64)
    pb = (pool_b.data_ptr() + (sb[:, None] * BR + np.arange(BR)[None, :]) * blk).astype(np.uint64)
    brv = C.c_ulonglong(BR)
    params = (X.GemmParam * batch)()
    base_pa, base_pb = pa.ctypes.data, pb.ctypes.data
    for t in range(batch):
        params[t].op.tertiary = C.addressof(brv)
        params[t].a.primary = base_pa + t * BR * 8; params[t].b.primary = base_pb + t * BR * 8
        params[t].c.primary = c.data_ptr() + t * M * N * 2
    plan = X.libxsmm_b200_gemm_plan_create(kernel, params, batch)
    assert plan and X.libxsmm_b200_gemm_plan_is_pooled(plan) == 1, "plan did not take the pooled tensor-core path"

    def step():
        assert X.libxsmm_b200_gemm_plan_run(plan) == 0
    step(); X.check()
    ha = pool_a.view(torch.int16).cpu().numpy().view(np.uint16); hb = pool_b.view(torch.int16).cpu().numpy().view(np.uint16)
    worst = 0.0
    for t in (0, 1, batch // 2, batch - 1):
        aa = (C.c_void_p * BR)(*[ha.ctypes.data + (int(sa[t]) * BR + r) * blk for r in range(BR)])
        ab = (C.c_void_p * BR)(*[hb.ctypes.data + (int(sb[t]) * BR + r) * blk for r in range(BR)])
        want = np.zeros(M * N, dtype=np.uint16)
        assert run_gemm(oracle, (M, N, K, M, K, M), (BF16, BF16, F32, BF16), FLAG_BETA_0, 1, 0, 0, BR, aa, ab, want) == 0
        got = c[t * M * N:(t + 1) * M * N].view(torch.int16).cpu().numpy().view(np.uint16)
        err = gen.normf_rel(gen.to_f64(want, BF16), gen.to_f64(got, BF16))
        assert err <= 5e-3, "mode R output differs from the oracle (tile %d, err %g)" % (t, err)
        worst = max(worst, err)
    total_ms, per = time_steps(torch, step, args.steps if full else max(5, args.steps), 3)
    X.check()
    if full:
        dump_outputs(args, torch, c=c)
    ms = sorted(per)[len(per) // 2]
    X.libxsmm_b200_gemm_plan_destroy(plan)
    flops = 2.0 * M * N * K * BR * batch
    tf = flops / (ms * 1e-3) / 1e12
    return {"metric": "batched BRGEMM GFLOP/s, mode R (bf16 64^3 br=8, address batch-reduce, operand pool of %d block-sets, C bf16 unique)" % pool_sets,
            "value": flops / (ms * 1e-3) / 1e9, "unit": "GFLOP/s", "ms_per_step": ms, "oracle_check": {"tiles": 4, "max_normf_rel": worst},
            "roofline": {"bound": "tensor", "achieved": tf, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / pk["bf16_tflops"], "traffic": traffic("gemm_pool_kernel"),
                         "kernel": "gemm_pool_kernel (resident operand sets, two tiles per M=128 instruction)",
                         "note": "a 128x64x16 tcgen05.mma costs 48 cycles (profiles/r01_umma_cost.txt: max(N/2, 32+N/4)), i.e. 67 % of the nominal "
                                 "2.38 PFLOP/s at 1965 MHz = 95 % of the measured cuBLAS peak: the bound of this tile shape"},
            "config": {"workload": "configs[1] mode R: tiles draw their A and B block-sets from pools of %d (L2-resident); C %.0f MB per step" % (pool_sets, batch * M * N * 2 / 1e6)}}


def strong_scaling(X, torch, pk, args, dist, world, rank):
    """configs[3]/[2] as BASELINE.json words them: the FIXED job (BCSC m_blocks = 8192, fsspmdm N = 1e6) cut over the ranks with
    shard_range -- contiguous ranges, nothing exchanged on the data path. Every rank runs its range at the same time; the job time is
    the slowest rank's (barrier + max). The one optional collective -- gathering the C ranges into one buffer on every rank with NCCL
    over NVLink -- is timed separately."""
    from libxsmm_b200.shard import shard_range
    res = {"scaling": "strong", "ranks": world}
    b0, b1 = shard_range(8192, world, rank, granule=4)              # 4 m_blocks of 32 rows form one 128-row MMA group
    r = also_bcsc(X, torch, pk, args, mblocks=b1 - b0, dist=dist)
    job_flops = 2.0 * 32 * 8192 * 512 * 512
    res["bcsc"] = {"m_blocks_total": 8192, "m_blocks_this_rank": b1 - b0, "ms_per_step": r["ms_per_step"], "value": job_flops / (r["ms_per_step"] * 1e-3) / 1e9,
                   "unit": "GFLOP/s (dense-equivalent, whole job)", "hbm_frac_per_gpu": r["roofline"]["frac"], "oracle_check": r.get("oracle_check")}
    n0, n1 = shard_range(1000000, world, rank, granule=16)
    f = also_fsspmdm(X, torch, pk, args, n_cols=n1 - n0, dist=dist)
    res["fsspmdm"] = {"n_total": 1000000, "n_this_rank": n1 - n0, "ms_per_step": f["ms_per_step"], "value": 2.0 * f["nnz"] * 1000000 / (f["ms_per_step"] * 1e-3) / 1e9,
                      "unit": "GFLOP/s (sparse, whole job)", "hbm_frac_per_gpu": f["roofline"]["frac"], "oracle_check": f.get("oracle_check")}
    # the optional gather: every rank contributes its C range of the BCSC job (8192/world m_blocks x 32 x 512 bf16)
    shard = torch.empty((b1 - b0) * 32 * 512, dtype=torch.bfloat16, device="cuda")
    full = torch.empty(world * shard.numel(), dtype=torch.bfloat16, device="cuda")
    for _ in range(3):
        dist.all_gather_into_tensor(full, shard)
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        dist.all_gather_into_tensor(full, shard)
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gms = float(t.item())
    res["gather"] = {"collective": "ncclAllGather of the C ranges (torch.distributed all_gather_into_tensor)", "bytes_received_per_rank": int((world - 1) * shard.numel() * 2),
                     "ms": gms, "GBps_in_per_gpu": (world - 1) * shard.numel() * 2 / (gms * 1e-3) / 1e9}
    return res


def also_meltw(X, torch, pk, args, sizes=(4096, 8192)):
    """three mateltwise kernels at 4096 x 4096 (fits L2 for 4-byte data: an L2 number) and 8192 x 8192 (> L2: the HBM number):
    f32 transpose, bf16 NORM->VNNI2 pack, f32 column-sum; roofline = operand + result bytes"""
    F32_, BF16_ = 1, 2
    out = []
    for n in sizes:
        x32 = torch.randn(n * n, device="cuda"); y32 = torch.empty(n * n, device="cuda")
        x16 = torch.randn(n * n, device="cuda").bfloat16(); y16 = torch.empty(n * n, dtype=torch.bfloat16, device="cuda")
        r32 = torch.empty(n, device="cuda")
        cases_ = [("transpose f32", X.MELTW_TYPE_UNARY_TRANSFORM_NORM_TO_NORMT, 0, F32_, F32_, x32, y32, 8.0 * n * n),
                  ("norm->vnni2 bf16", X.MELTW_TYPE_UNARY_TRANSFORM_NORM_TO_VNNI2, 0, BF16_, BF16_, x16, y16, 4.0 * n * n),
                  ("reduce cols x_op_add f32", X.MELTW_TYPE_UNARY_REDUCE_X_OP_ADD, X.MELTW_FLAG_UNARY_REDUCE_COLS, F32_, F32_, x32, r32, 4.0 * n * n + 4.0 * n)]
        for name, op, flags, tin, tout, src, dst, nbytes in cases_:
            k = X.libxsmm_dispatch_meltw_unary(op, X.libxsmm_create_meltw_unary_shape(n, n, n, n, tin, tout, F32_), flags)
            if not k:
                out.append({"op": name, "n": n, "error": "dispatch returned NULL"}); continue
            p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = src.data_ptr(), dst.data_ptr()
            fn = X.MELTW_UNARY_FN(k)

            def step():
                fn(C.byref(p))
            step(); X.check()
            if name.startswith("transpose"):
                assert torch.equal(dst.view(n, n)[:96, -96:], src.view(n, n).t()[:96, -96:]), "transpose check"
            elif name.startswith("norm->vnni2"):
                want = src.view(n, n)[:64].view(32, 2, n).permute(0, 2, 1).reshape(-1)      # [n/2][m][2] <- [n][m]
                assert torch.equal(dst[:64 * n], want), "vnni2 pack check"
            else:
                want = src.view(n, n).sum(0)
                assert torch.allclose(dst, want, rtol=1e-3, atol=2e-2), "column-sum check"
            total_ms, per = time_steps(torch, step, max(5, args.steps // 2), 3)
            X.check()
            ms = sorted(per)[len(per) // 2]
            gbs = nbytes / (ms * 1e-3) / 1e9
            out.append({"op": name, "n": n, "ms": ms, "GBps": gbs, "hbm_frac": gbs / pk["hbm_gbs"], "algorithmic_bytes": nbytes,
                        "l2_note": "" if nbytes > 2.5e8 else "operands fit L2: not an HBM number"})
        del x32, y32, x16, y16, r32
    return {"metric": "mateltwise GB/s at 4096^2 and 8192^2", "points": out}


# ------------------------------------------------------------------------------------------------ CPU side
def physical_cores():
    """one logical CPU per physical core among those this process may run on (/proc/cpuinfo: physical id, core id)"""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except Exception:
        allowed = list(range(os.cpu_count() or 1))
    seen, cur = {}, {}
    try:
        with open("/proc/cpuinfo") as f:
            for line in f.read().split("\n") + [""]:
                if ":" in line:
                    k, v = [x.strip() for x in line.split(":", 1)]
                    cur[k] = v
                elif cur:
                    cpu = int(cur.get("processor", -1))
                    key = (cur.get("physical id", "0"), cur.get("core id", str(cpu)))
                    if cpu in allowed and key not in seen:
                        seen[key] = cpu
                    cur = {}
    except Exception:
        pass
    return sorted(seen.values()) or allowed


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every PHYSICAL core this process may run on, one
    pinned thread per core (hyper-threads share the AMX unit and only add noise). Must run before the OpenMP runtime of
    oracle/_ref is loaded."""
    cores = physical_cores()
    try:
        os.sched_setaffinity(0, set(cores))
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(len(cores))
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    return len(cores)


def host_mem_available_gb():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable"):
                    return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 8.0


def cpu_brgemm_passes(warm, passes, want_tiles=BATCH):
    """`passes` timed passes of the reference's JIT over the strided batch, buffers owned and first-touched by the OpenMP
    threads of oracle/_ref (ref_bench_brgemm_owned). The sample is the full batch when the host can hold it (9.7 GB),
    else the largest power-of-two fraction that fits a third of the available memory (never below 8192 tiles = 1.2 GB,
    several times the box's cache)."""
    ncores = use_all_host_threads()
    from oracle_ffi import ref_lib
    if ref_lib is None:
        return None, {"value": None, "unit": "GFLOP/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref/libxsmm_ref.so missing"}
    per_tile = (2 * BR * M * K + 2 * BR * K * N + 4 * M * N)
    tiles = want_tiles
    while tiles > 8192 and tiles * per_tile / 1e9 > host_mem_available_gb() / 3:
        tiles //= 2
    fn = ref_lib.ref_bench_brgemm_owned
    fn.restype = C.c_int
    fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_ulonglong, C.c_uint, C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_double)]
    secs = (C.c_double * passes)()
    is_ref, chk = C.c_int(0), C.c_double(0)
    flags = FLAG_BETA_0 | 256   # VNNI_A: the layout the reference's x86 bf16 JIT (AMX/AVX-512 BF16) is written for
    rc = fn(M, N, K, BR, flags, tiles, warm, passes, secs, C.byref(is_ref), C.byref(chk))
    if rc != 0:
        return None, {"value": None, "unit": "GFLOP/s", "cores": ncores, "kind": "reference",
                      "sample": "JIT dispatch returned NULL on this host" if rc == -1 else "host cannot hold the sample"}
    fl = 2.0 * M * N * K * BR * tiles
    gf = sorted(fl / t / 1e9 for t in secs)
    info = {"value": gf[len(gf) // 2], "unit": "GFLOP/s", "cores": ncores, "kind": "reference", "min": gf[0], "max": gf[-1], "passes": passes,
            "sample": "%d of %d tiles (%.1f GB of A+B+C, every operand unique, first-touched by the thread that streams it) x %d passes after %d warm-up, "
                      "one pinned OpenMP thread per physical core (OMP_PLACES=cores, close), LIBXSMM JIT target %s%s, VNNI_A layout; value = median pass" % (
                          tiles, want_tiles, tiles * per_tile / 1e9, passes, warm, ref_lib.ref_target_arch().decode(), " [C reference kernel!]" if is_ref.value else "")}
    return [float(t) for t in secs], info


def cpu_baseline_brgemm(passes=5):
    """the reference's own JIT BRGEMM kernel over the same batch on the host cores: a bounded number of passes"""
    return cpu_brgemm_passes(1, passes)[1]


def cpu_baseline_fsspmdm(a_dense, Mf, Kf, nnz, n_sample=200000, budget_s=4.0):
    """the reference's fsspmdm JIT on a bounded N-slice of the same operator, all host cores (slices of N per thread)"""
    import numpy as np
    use_all_host_threads()
    from oracle_ffi import ref_lib
    if ref_lib is None:
        return {"value": None, "unit": "GFLOP/s (sparse)", "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}
    rng = np.random.default_rng(7)
    b = rng.standard_normal(Kf * n_sample).astype(np.float32); c = np.zeros(Mf * n_sample, dtype=np.float32)
    one = np.array([1.0], dtype=np.float32); zero = np.array([0.0], dtype=np.float32)
    args = (F32, Mf, n_sample, Kf, Kf, one.ctypes.data, zero.ctypes.data, a_dense.ctypes.data, b.ctypes.data, c.ctypes.data)
    t1 = ref_lib.ref_bench_fsspmdm(*args, 1)
    if t1 < 0:
        return {"value": None, "unit": "GFLOP/s (sparse)", "cores": int(ref_lib.ref_max_threads()), "kind": "reference", "sample": "create returned NULL"}
    reps = max(1, min(500, int(budget_s / max(t1, 1e-4))))
    t = ref_lib.ref_bench_fsspmdm(*args, reps)
    return {"value": 2.0 * nnz * n_sample * reps / t / 1e9, "unit": "GFLOP/s (sparse)", "gbs": 4.0 * (Kf + Mf) * n_sample * reps / t / 1e9,
            "cores": int(ref_lib.ref_max_threads()), "kind": "reference", "sample": "N=%d columns (%.0f MB of B+C) x %d passes, LIBXSMM JIT" % (n_sample, 4.0 * (Kf + Mf) * n_sample / 1e6, reps)}


def cpu_baseline_bcsc(colptr, rowidx, nnzb, geo, mblocks=1024, budget_s=4.0):
    """the reference's BCSC JIT (AMX on SPR) on a bounded number of m_blocks, contiguous ranges per thread"""
    import numpy as np
    use_all_host_threads()
    from oracle_ffi import ref_lib, iarr
    Mb, Kb, Nb, bk, bn = geo
    if ref_lib is None:
        return {"value": None, "unit": "GFLOP/s (dense-equivalent)", "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}
    rng = np.random.default_rng(8)

    def bf16(n):
        x = (rng.integers(-5, 6, size=n).astype(np.float32) / 10).view(np.uint32)
        return ((x + 0x7FFF + ((x >> 16) & 1)) >> 16).astype(np.uint16)
    a = bf16(mblocks * Kb * Mb); bv = bf16(nnzb * bk * bn); c = np.zeros(mblocks * Nb * Mb, dtype=np.uint16)
    cp = colptr.copy(); ri = rowidx.copy()
    args = (iarr(BF16, BF16, F32, BF16), iarr(mblocks, Mb, Kb, Nb, bk, bn), FLAG_BETA_0 | 256, a.ctypes.data, bv.ctypes.data, cp.ctypes.data, ri.ctypes.data, c.ctypes.data)
    t1 = ref_lib.ref_bench_bcsc(*args, 1)
    if t1 < 0:
        return {"value": None, "unit": "GFLOP/s (dense-equivalent)", "cores": int(ref_lib.ref_max_threads()), "kind": "reference", "sample": "JIT returned NULL on this host"}
    reps = max(1, min(500, int(budget_s / max(t1, 1e-4))))
    t = ref_lib.ref_bench_bcsc(*args, reps)
    return {"value": 2.0 * Mb * mblocks * Nb * Kb * reps / t / 1e9, "unit": "GFLOP/s (dense-equivalent)", "cores": int(ref_lib.ref_max_threads()), "kind": "reference",
            "sample": "%d m_blocks (%.0f MB of A+C) x %d passes, LIBXSMM JIT target %s" % (mblocks, 4.0 * mblocks * Mb * (Kb + Nb) / 2 / 1e6, reps, ref_lib.ref_target_arch().decode())}


def run_reference(args):
    """Reference arm: a step is one pass of the reference's JIT kernel over the strided batch on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps = max(1, args.steps)
    secs, info = cpu_brgemm_passes(max(1, args.warmup), steps)
    if secs is None:
        print(json.dumps({"impl": "reference", "unavailable": info["sample"]}))
        return
    v = info["value"]
    print(json.dumps({"impl": "reference", "metric": METRIC,
                      "value": v, "unit": "GFLOP/s", "n_gpus": world, "steps": steps, "warmup": max(1, args.warmup),
                      "ms_per_step": sum(secs) / len(secs) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH,
                                 "reference_arm": "host CPU (not scaled with --gpus): LIBXSMM JIT through libxsmm_dispatch_brgemm, OpenMP over tiles; " + info["sample"]},
                      "cpu_baseline": info,
                      "e2e": {"value": v, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="brgemm", choices=["brgemm", "brgemm_r", "fsspmdm", "bcsc", "sweep"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed path's last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
