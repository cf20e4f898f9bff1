#!/usr/bin/env python
"""bench.py — rows/s of the headline workload (2-D 1024^2 count over fp32 x,y; limits [-3,3]) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (default N=1)
    python bench.py --impl reference --steps K --warmup W     # the reference's own CPU superagg on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR   # also write the last timed step's grid to DIR/count.npy

One "step" = one pass of the hot path over the whole synthetic batch (rows_per_gpu rows on every rank):
reset grid -> fused binby kernel -> (N>1) NCCL all-reduce of the 1027^2 int64 grid -> D2H of the grid.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPE = 1024
LIMITS = (-3.0, 3.0)
BYTES_PER_ROW = 8  # algorithmic: x and y, fp32 each (SURVEY.md section 8d)
METRIC = "rows/s 2D 1024^2 count on fp32 (binby x,y; limits [-3,3])"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=float, default=1e9, help="rows per GPU (weak scaling)")
    ap.add_argument("--e2e-rows", type=float, default=float(1 << 28), help="rows per GPU per step of the host-buffer (e2e) leg")
    ap.add_argument("--e2e-chunk", type=float, default=float(1 << 24))
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-threads", type=int, default=16, help="Python feeder threads of the e2e leg (the executor's thread pool)")
    ap.add_argument("--cpu-rows", type=float, default=0, help="rows of the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="serialise every step's all-reduce + D2H behind its kernels (default: they run on a second stream under the next step)")
    ap.add_argument("--no-also", action="store_true", help="skip the other BASELINE.json configs (sum, 3-D mean+std, groupby)")
    ap.add_argument("--also-sample", type=float, default=1e8, help="rows of the parity sample of each `also` config against oracle/_ref")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the count grid of the last timed step to DIR/count.npy (float64, the shape "
                                                          "get_result() returns), to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed: use it with --impl b200")
    return args


def dump_outputs(path, arrays):
    """one <name>.npy per array, as float64 (exact for counts below 2^53)"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index, period=0.005):
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = threading.Event()
        self.err = None
        self.nv = self.h = None
        try:  # NVML is initialised BEFORE the timed region so that the first sample lands inside it
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.err = repr(e)

    def run(self):
        nv, h = self.nv, self.h
        if nv is None:
            return
        try:
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            while True:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                if self.stop_flag.wait(self.period):
                    break
        except Exception as e:
            self.err = repr(e)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "error": self.err}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(x, y, nthreads):
    """The reference's own CPU path on host arrays: compiled unmodified superagg (oracle/_ref) driven by the restated
    executor chunk loop; falls back to the C port (1 thread) only if the compiled reference is absent."""
    from oracle import oracle as O, ref_driver as R
    n = len(x)
    binners = [O.scalar(x, LIMITS[0], LIMITS[1], SHAPE), O.scalar(y, LIMITS[0], LIMITS[1], SHAPE)]
    aggs = [O.agg("count")]
    if R.available():
        t0 = time.perf_counter()
        job = R.RefBinby(binners, aggs, nthreads)
        res = job.run(n)
        dt = time.perf_counter() - t0
        return res[0], dt, "reference", nthreads
    t0 = time.perf_counter()
    res = O.binby(binners, aggs, n)
    dt = time.perf_counter() - t0
    return res[0], dt, "port", 1


def cpu_calibrated_rows(nthreads, target_s=2.5):
    import numpy as np
    rng = np.random.default_rng(1)
    n = 4_000_000
    x = rng.standard_normal(n, dtype=np.float32)
    y = rng.standard_normal(n, dtype=np.float32)
    cpu_reference_run(x, y, nthreads)
    _, dt, _, _ = cpu_reference_run(x, y, nthreads)
    rate = n / dt
    rows = int(min(4e8, max(1e7, rate * target_s)))
    return rows


def gen_host(n, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(n, dtype=np.float32)
    y = rng.standard_normal(n, dtype=np.float32)
    return x, y


def run_reference(args):
    """--impl reference: the reference CPU implementation, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nthreads = os.cpu_count() or 1
    rows = int(args.cpu_rows) or cpu_calibrated_rows(nthreads)
    x, y = gen_host(rows, 42)
    for _ in range(args.warmup):
        cpu_reference_run(x, y, nthreads)
    t = 0.0
    kind = cores = None
    for _ in range(args.steps):
        _, dt, kind, cores = cpu_reference_run(x, y, nthreads)
        t += dt
    value = rows * args.steps / t
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"df.count(binby=[x,y], limits=[[-3,3]]*2, shape=1024) on {rows:.3g} fp32 rows per step (bounded sample), host CPU"},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": kind,
                         "sample": f"{rows} rows/step, N(0,1) fp32 x,y, seed 42, executor chunking restated (1M-row chunks)", "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
def timed_ms(stream, ctx, fn, reps):
    """mean device time of `fn` (launches on the slot stream) over `reps` runs after one warm-up; CUDA events on that stream"""
    import torch
    fn()
    ctx.sync(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    ctx.sync(0)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def also_configs(args, ctx, stream, gen, peak, rows, nthreads):
    """BASELINE.json configs[1..3] at full size (device-resident, timed with CUDA events) + a parity check of the first
    `--also-sample` rows against the compiled, unmodified reference (oracle/_ref) run on the host cores."""
    import numpy as np
    import torch
    from oracle import oracle as O, ref_driver as R
    from vaex_b200 import superagg, superutils
    out = {}
    ns = int(min(args.also_sample, rows))
    have_ref = R.available()

    def entry(ms, bytes_per_row, kernel, parity, **extra):
        gbs = bytes_per_row * rows / (ms * 1e-3) / 1e9
        return dict(rows=rows, rows_per_s=rows / (ms * 1e-3), ms_per_step=ms, algorithmic_bytes_per_row=bytes_per_row, achieved_gbs=gbs,
                    frac=gbs / peak, kernel=kernel, parity=parity, parity_against="oracle/_ref (compiled reference), %d threads" % nthreads if have_ref else "unavailable",
                    parity_rows=ns, **extra)

    # ---- configs[1]: df.sum(z, binby=[x,y], shape=1024) on fp32 ---------------------------------------------------------------
    x = torch.empty(rows, dtype=torch.float32, device="cuda").normal_(generator=gen)
    y = torch.empty(rows, dtype=torch.float32, device="cuda").normal_(generator=gen)
    z = torch.empty(rows, dtype=torch.float32, device="cuda").normal_(generator=gen)
    bx = superagg.BinnerScalar_float32(1, "x", LIMITS[0], LIMITS[1], SHAPE)
    by = superagg.BinnerScalar_float32(1, "y", LIMITS[0], LIMITS[1], SHAPE)
    grid = superagg.Grid([bx, by])
    asum = superagg.AggSum_float32(grid, 1, 1)

    def bind(n):
        bx.set_data(0, x[:n])
        by.set_data(0, y[:n])
        asum.set_data(0, z[:n], 0)

    def c2():
        asum.reset(0)
        grid.bin(0, [asum], rows)
    bind(rows)
    ms = timed_ms(stream, ctx, c2, 3)
    parity = None
    if have_ref:
        bind(ns)
        asum.reset(0)
        grid.bin(0, [asum], ns)
        got = asum.get_result()
        xc, yc, zc = (t[:ns].cpu().numpy() for t in (x, y, z))
        want = R.RefBinby([O.scalar(xc, LIMITS[0], LIMITS[1], SHAPE), O.scalar(yc, LIMITS[0], LIMITS[1], SHAPE)], [O.agg("sum", zc)], nthreads).run(ns)[0]
        parity = bool(np.allclose(got, want, rtol=1e-6, atol=1e-9 * float(np.abs(want).max())))
    out["configs[1] df.sum(z, binby=[x,y], shape=1024), 1e9 fp32 rows"] = entry(ms, 12, "k_binby_fast<float,2,float> (one RED.ADD.F64 per row)", parity, tolerance="rtol 1e-6")
    del x, y, z, bx, by, grid, asum
    torch.cuda.empty_cache()

    # ---- configs[2]: df.mean(v) + df.std(v), binby=[x,y,z], shape=256 on fp64: count, sum, sum^2 fused -----------------------------
    cols = [torch.empty(rows, dtype=torch.float64, device="cuda").normal_(generator=gen) for _ in range(4)]
    bs = [superagg.BinnerScalar_float64(1, "xyz"[i], LIMITS[0], LIMITS[1], 256) for i in range(3)]
    grid = superagg.Grid(bs)
    aggs = [superagg.AggCount_float64(grid, 1, 1), superagg.AggSum_float64(grid, 1, 1), superagg.AggSumMoment_float64(grid, 1, 1, 2)]

    def bind3(n):
        for b, c in zip(bs, cols):
            b.set_data(0, c[:n])
        for a in aggs:
            a.set_data(0, cols[3][:n], 0)

    def c3():
        for a in aggs:
            a.reset(0)
        grid.bin(0, aggs, rows)
    bind3(rows)
    ms = timed_ms(stream, ctx, c3, 2)
    parity = None
    if have_ref:
        bind3(ns)
        for a in aggs:
            a.reset(0)
        grid.bin(0, aggs, ns)
        got = [a.get_result() for a in aggs]
        hc = [c[:ns].cpu().numpy() for c in cols]
        want = R.RefBinby([O.scalar(hc[i], LIMITS[0], LIMITS[1], 256) for i in range(3)],
                          [O.agg("count", hc[3]), O.agg("sum", hc[3]), O.agg("sum_moment", hc[3], moment=2)], nthreads).run(ns)
        parity = bool(np.array_equal(got[0], want[0]) and all(np.allclose(got[k], want[k], rtol=1e-6, atol=1e-9 * float(np.abs(want[k]).max())) for k in (1, 2)))
        del hc, want
    out["configs[2] df.mean(v)+df.std(v), binby=[x,y,z], shape=256, 1e9 fp64 rows"] = entry(
        ms, 32, "k_sort_partition + k_sort_apply (region-sorted scatter, csrc/tilesort.cu)", parity, tolerance="count bit-exact; sum, sum^2 rtol 1e-6", grid_cells=len(grid))
    del cols, bs, grid, aggs
    torch.cuda.empty_cache()

    # ---- configs[3]: df.groupby(k).agg({v: [sum, count]}), 1e6 sparse int64 keys ------------------------------------------------
    keys = torch.randint(0, 1_000_000, (rows,), device="cuda", dtype=torch.int64, generator=gen) * 256 + 5
    v = torch.empty(rows, dtype=torch.float64, device="cuda").normal_(generator=gen)
    torch.cuda.synchronize()

    def groupby(n, time_it):
        k, vv = keys[:n], v[:n]
        ctx.sync(0)
        t0 = time.perf_counter()
        s = superutils.ordered_set_int64(7)
        s.update(k, -1)
        nkeys = len(s)  # finalises: ordinals are defined
        ctx.sync(0)
        t1 = time.perf_counter() - t0
        hb = superagg.BinnerHash_int64(1, "k", s)
        g = superagg.Grid([hb])
        hb.set_data(0, k)
        a_sum, a_cnt = superagg.AggSum_float64(g, 1, 1), superagg.AggCount_float64(g, 1, 1)
        for a in (a_sum, a_cnt):
            a.set_data(0, vv, 0)

        def p2():
            a_sum.reset(0)
            a_cnt.reset(0)
            g.bin(0, [a_sum, a_cnt], n)
        ms2 = timed_ms(stream, ctx, p2, 2) if time_it else (p2(), 0.0)[1]
        return s, nkeys, t1 * 1e3, ms2, a_sum.get_result(), a_cnt.get_result()
    groupby(rows, False)  # first build grows the table: keep it out of the timing, like the other configs' warm-up
    s, nkeys, ms1, ms2, _, gcnt = groupby(rows, True)
    assert int(gcnt.sum()) == rows
    parity = None
    if have_ref:
        s, nk, _, _, gsum, gcnt = groupby(ns, False)
        gk = s.key_array()
        hk, hv = keys[:ns].cpu().numpy(), v[:ns].cpu().numpy()
        rk, rsum, rcnt = R.groupby_sum_count(hk, hv, nthreads)
        # the reference's ordinals depend on thread timing (SURVEY section 7): compare as key -> (sum, count) maps
        og, orf = np.argsort(gk), np.argsort(rk)
        parity = bool(len(gk) == len(rk) and np.array_equal(gk[og], rk[orf]) and np.array_equal(np.asarray(gcnt)[:nk][og], np.asarray(rcnt)[:len(rk)][orf])
                      and np.allclose(np.asarray(gsum)[:nk][og], np.asarray(rsum)[:len(rk)][orf], rtol=1e-6, atol=1e-9))
    e = entry(ms1 + ms2, 24, "k_set_insert + finalise (pass 1), fused hash-probe binner k_binby (pass 2)", parity, tolerance="keys and counts bit-exact; sums rtol 1e-6",
              unique_keys=nkeys, pass1_ms=ms1, pass2_ms=ms2, pass1_note="wall clock incl. finalisation (ordinals defined), table already grown")
    out["configs[3] df.groupby(k).agg({v:[sum,count]}), 1e6 sparse int64 keys, 1e9 rows"] = e
    del keys, v
    torch.cuda.empty_cache()
    return out


def e2e_leg(args, ctx, world, rank, local, x, y, barrier, sampler, out):
    """End to end through the reference-facing front: PAGEABLE numpy columns -> Frame.count(binby=...) -> chunk-feed loop on T
    Python threads -> TaskPartAggregation.process(thread_index, i1, i2, ..., blocks) -> b200_bin(HOST) on slot thread_index ->
    (N>1: NCCL all-reduce) -> numpy result.  Host->device copies of every chunk and the device->host read of the grid are inside
    the timed region (wall clock, max over ranks).  Timed with vaex's chunk cap (1M rows, vaex/settings.py:85-87) — the headline
    `value` — and with 16M-row chunks; the pinned + B200_FLAG_ASYNC_HOST figure through the native class protocol (B2) is kept as
    a third key."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from vaex_b200 import _lib, engine, execution, superagg
    from vaex_b200.frame import Frame
    erows = int(args.e2e_rows)
    xn = x[:erows].cpu().numpy()  # plain pageable host memory, what a numpy / memory-mapped vaex column is
    yn = y[:erows].cpu().numpy()
    nthreads = max(1, min(args.e2e_threads, (os.cpu_count() or 8) // max(world, 1)))
    cells = (SHAPE + 3) ** 2
    res = {}

    def run(chunk_max, steps):
        ex = execution.Executor(nthreads=nthreads, chunk_size_max=chunk_max)
        df = Frame({"x": xn, "y": yn}, executor=ex)

        def one():
            g = df.count(binby=["x", "y"], limits=[list(LIMITS), list(LIMITS)], shape=SHAPE, edges=True)
            if world > 1:
                t = torch.from_numpy(np.ascontiguousarray(g)).cuda()
                dist.all_reduce(t)
                g = t.cpu().numpy()
            return g
        one()  # warm-up: both bounce buffers of every slot and the arenas are allocated here
        one()
        barrier()
        w0 = time.perf_counter()
        for _ in range(steps):
            g = one()
        barrier()
        w = time.perf_counter() - w0
        if world > 1:
            t = torch.tensor([w], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            w = float(t.item())
        assert int(g.sum()) == erows * world, "row conservation failed in the e2e leg"
        return erows * world * steps / w, ex.chunk_size_for(erows)

    sampler2 = ClockSampler(local, period=0.05)  # NVML queries take driver locks the 16 feeder threads need: poll gently
    sampler2.start()
    v1, c1 = run(1 << 20, args.e2e_steps)
    v16, c16 = run(1 << 24, args.e2e_steps)
    c2 = sampler2.result()
    if c2.get("sm_mhz") is not None:  # the e2e steps are a timed region too: fold their clock samples in
        both = sorted(sampler.samples + sampler2.samples)
        out["clocks"] = {"sm_mhz": both[len(both) // 2], "sm_max_mhz": c2["sm_max_mhz"], "reasons": sorted(set(out["clocks"]["reasons"]) | set(c2["reasons"])),
                         "samples": len(both), "windows": "device-resident steps + e2e steps"}
    res = {"value": v1, "unit": "rows/s", "h2d_bytes_per_step": erows * BYTES_PER_ROW, "d2h_bytes_per_step": cells * 8, "rows_per_step_per_gpu": erows,
           "chunk_rows": c1, "threads": nthreads,
           "path": "pageable numpy -> Frame.count -> TaskPartAggregation.process -> b200_bin(HOST): page-locked bounce ring, no per-call sync",
           "chunks_16M": {"value": v16, "unit": "rows/s", "chunk_rows": c16}}

    # the plumbing ceiling: pinned host columns through the native class protocol with B200_FLAG_ASYNC_HOST on 4 slots
    bx = superagg.BinnerScalar_float32(4, "x", LIMITS[0], LIMITS[1], SHAPE)
    by = superagg.BinnerScalar_float32(4, "y", LIMITS[0], LIMITS[1], SHAPE)
    grid = superagg.Grid([bx, by])
    agg = superagg.AggCount_int64(grid, 1, 4)
    host_grid = torch.empty(cells, dtype=torch.int64).pin_memory()
    xh, yh = torch.from_numpy(xn).pin_memory(), torch.from_numpy(yn).pin_memory()
    xp, yp = xh.numpy(), yh.numpy()
    chunk, nslots = int(args.e2e_chunk), 4

    def pinned_step():
        agg.reset(0)
        ctx.sync(0)
        for c, i1 in enumerate(range(0, erows, chunk)):
            i2 = min(i1 + chunk, erows)
            sl = c % nslots
            bx.set_data(sl, xp[i1:i2])
            by.set_data(sl, yp[i1:i2])
            grid.bin(sl, [agg], i2 - i1, row_offset=i1, flags=_lib.FLAG_ASYNC_HOST)
        ctx.sync(-1)
        if world > 1:
            engine.all_reduce([agg], slot=0)
        agg.read_async(0, host_grid)
        ctx.sync(0)
    pinned_step()
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        pinned_step()
    barrier()
    w = time.perf_counter() - w0
    if world > 1:
        t = torch.tensor([w], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        w = float(t.item())
    assert int(host_grid.sum().item()) == erows * world
    res["pinned_async_b2"] = {"value": erows * world * args.e2e_steps / w, "unit": "rows/s", "chunk_rows": chunk, "slots": nslots,
                              "note": "pre-pinned host columns -> b200_bin(HOST, ASYNC) on 4 slots: the PCIe ceiling of this path"}
    return res


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun the way the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a GPU: vaex_b200 has no CPU fallback (use --impl reference for the CPU reference)")
    torch.cuda.set_device(local)
    os.environ["VAEX_B200_DEVICE"] = str(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    from vaex_b200 import _lib, engine, superagg

    ctx = _lib.context(local)
    rows = int(args.rows)
    gen = torch.Generator(device="cuda").manual_seed(42 + rank)
    x = torch.empty(rows, dtype=torch.float32, device="cuda").normal_(generator=gen)
    y = torch.empty(rows, dtype=torch.float32, device="cuda").normal_(generator=gen)

    bx = superagg.BinnerScalar_float32(4, "x", LIMITS[0], LIMITS[1], SHAPE)
    by = superagg.BinnerScalar_float32(4, "y", LIMITS[0], LIMITS[1], SHAPE)
    grid = superagg.Grid([bx, by])
    # df.count() == count('*'): dtype_in int64, no data column (vaex/agg.py:254-257).  TWO grids: step k bins into grid k%2 on slot 0's
    # stream while grid (k-1)%2 is all-reduced over NVLink and copied to the host on slot 1's stream — the per-step tail
    # (NCCL all-reduce of 8.4 MB + 8.4 MB D2H) hides behind the next step's kernels (--no-overlap serialises it again).
    aggs = [superagg.AggCount_int64(grid, 1, 4) for _ in range(2)]
    cells = len(grid)
    host_grids = [torch.empty(cells, dtype=torch.int64).pin_memory() for _ in range(2)]
    stream = engine.slot_stream(ctx, 0)
    tail_slot = 0 if args.no_overlap else 1
    tail_stream = engine.slot_stream(ctx, tail_slot)
    tail_done = [None, None]
    bx.set_data(0, x)
    by.set_data(0, y)

    kernel_ms = []
    nstep = [0]

    def step(timed):
        k = nstep[0] % 2
        nstep[0] += 1
        agg = aggs[k]
        if tail_done[k] is not None and tail_slot != 0:
            stream.wait_event(tail_done[k])  # grid k is free again once its previous tail has read it
        agg.reset(0)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        grid.bin(0, [agg], rows)
        e1.record(stream)
        if tail_slot != 0:
            tail_stream.wait_event(e1)
        if world > 1:
            engine.all_reduce([agg], slot=tail_slot)
        agg.read_async(tail_slot, host_grids[k])
        if tail_slot != 0:
            tail_done[k] = torch.cuda.Event()
            tail_done[k].record(tail_stream)
        if timed:
            kernel_ms.append((e0, e1))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(False)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(args.steps):
        step(True)
    stream.wait_event(tail_done[(nstep[0] - 1) % 2]) if tail_slot != 0 else None  # the timed region ends when the LAST step's result is on the host
    t1.record(stream)
    barrier()
    clocks = sampler.result()
    total_ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([total_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    kms = sum(a.elapsed_time(b) for a, b in kernel_ms) / len(kernel_ms)
    agg = aggs[0]
    for hg in host_grids[: min(2, nstep[0])]:
        counted = int(hg.sum().item())
        assert counted == rows * world, f"row conservation failed: grid holds {counted}, expected {rows * world}"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"count": host_grids[(nstep[0] - 1) % 2].numpy().reshape(grid.shapes, order="F")})

    value = rows * world * args.steps / (total_ms * 1e-3)
    # count(*) on a 1027^2 grid takes the ring-partition path from 2^22 rows: 2 kernels (+ 2 memsets) per batch of <= 2^30 rows
    ring = rows >= (1 << 22)
    nbatch = (rows + (1 << 30) - 1) >> 30
    launches_per_step = 2 * nbatch if ring else 1
    peak, peak_src = measured_peak()
    achieved = BYTES_PER_ROW * rows / (kms * 1e-3) / 1e9
    # DRAM traffic of the timed build, from the kernels' own counters (b200_ctx_path_stats): every row's keys are read once
    # (8 B), every 16-bit scratch entry is written once by k_ring_partition and read once by k_ring_count, plus the list tables
    # that are memset before the pass; the grid (8.4 MB) stays in the L2.  profiles/r02_ncu_ring_v5.txt has the profiler's view of
    # the same pair (dram__bytes 12.0 B/row).
    st = ctx.path_stats(0) if ring else None
    traffic = None
    if st and st["rows"]:
        per_batch = st["rows"] * BYTES_PER_ROW + st["entries"] * 2 * 2 + st["memset_bytes"]
        traffic = per_batch * rows / st["rows"] / 1e9

    out = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"df.count(binby=[x,y], limits=[[-3,3]]*2, shape=1024) on {rows:.4g} fp32 rows per GPU, device-resident columns"
                               + (" = BASELINE configs[4] (1e10 rows over 8 GPUs)" if world == 8 and rows == 1_250_000_000 else ""),
                   "rows_per_gpu": rows, "grid_cells": cells, "parallelism": f"row-shard x{world} + NCCL all-reduce of the int64 grid",
                   "step_tail": "serialised" if args.no_overlap else "all-reduce + D2H of step k on a second stream under the kernels of step k+1 (two grids)",
                   "l2": "inputs (8 GB/GPU) far exceed L2; no flush needed", "index_math": "fp64, bit-exact with the reference"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_unit": "GB per step",
                     "traffic_source": "counters of the timed build (b200_ctx_path_stats): 8 B/row keys + 2 x 2 B per scratch entry + memsets" if traffic else None,
                     "scratch_entries_per_row": (st["entries"] / st["rows"]) if st and st["rows"] else None,
                     "peak_source": peak_src, "kernel": "k_ring_partition<float,2> + k_ring_count (csrc/ringcount.cu)" if ring else "k_binby_fast",
                     "kernel_ms": kms, "algorithmic_bytes_per_row": BYTES_PER_ROW, "launches_per_step": launches_per_step,
                     "note": "achieved = 8 B/row x rows per step / device time of the step's binby launches (CUDA events on the launching "
                             "stream); both kernels are bound by shared-memory atomic throughput (one ATOMS per row each), see DESIGN.md section 4"},
        "gpu_launches": args.steps * launches_per_step,
        "clocks": clocks,
    }

    # ---- e2e: host buffers through the reference-facing task part, H2D inside the timed region ------------------------------
    if not args.no_e2e:
        out["e2e"] = e2e_leg(args, ctx, world, rank, local, x, y, barrier, sampler, out)

    # ---- CPU baseline (rank 0, N=1 only): the compiled reference on the host cores, bounded sample -------------------
    if rank == 0 and world == 1 and not args.no_cpu:
        nthreads = os.cpu_count() or 1
        crows = int(args.cpu_rows) or cpu_calibrated_rows(nthreads, target_s=4.0)
        crows = min(crows, rows)
        xc = x[:crows].cpu().numpy()
        yc = y[:crows].cpu().numpy()
        cpu_reference_run(xc, yc, nthreads)
        best = None
        cgrid = None
        for _ in range(3):
            cgrid, dt, kind, cores = cpu_reference_run(xc, yc, nthreads)
            best = dt if best is None else min(best, dt)
        # the same code on ONE thread (BASELINE.md section 3), on a smaller sample
        r1 = min(crows, 20_000_000)
        _, dt1, _, _ = cpu_reference_run(xc[:r1], yc[:r1], 1)
        # parity on the sample while we are here: the GPU grid for the same rows must be bit-identical
        agg.reset()
        bx.set_data(0, x[:crows])
        by.set_data(0, y[:crows])
        grid.bin(0, [agg], crows)
        ggrid = agg.get_result()
        out["cpu_baseline"] = {"value": crows / best, "unit": "rows/s", "cores": cores, "kind": kind, "host_cpus": os.cpu_count(),
                               "sample": f"first {crows} rows of the GPU arrays, best of 3, executor chunk loop restated (1M-row chunks), includes get_result fold",
                               "one_thread": {"value": r1 / dt1, "unit": "rows/s", "cores": 1, "sample": f"first {r1} rows"},
                               "parity_on_sample": bool(np.array_equal(np.asarray(cgrid), ggrid))}
        out["config"]["cpu_baseline_sample_rows"] = crows
        del xc, yc

    # ---- the other BASELINE.json configurations at full size, each with a parity check against the compiled reference --------
    if rank == 0 and world == 1 and not args.no_also:
        del x, y, bx, by, grid, agg, aggs
        torch.cuda.empty_cache()
        out["also"] = also_configs(args, ctx, stream, gen, peak, rows, os.cpu_count() or 1)

    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
