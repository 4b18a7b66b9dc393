#!/usr/bin/env python3
"""Headline benchmark: norm.coex on 100k cells x 20k genes (BASELINE.json metric), one process
per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the hot path over the synthetic matrix: residualise + quantise, (N > 1:
all-gather of the digit planes), tensor-core contraction with the fused r / P epilogue.
  value  unique gene pairs per second with inputs and outputs resident in HBM;
  e2e    the same pairs through the public API with HOST buffers: pinned host -> device copy of
         the expression matrix and device -> pinned host copy of P and dot inside the timed region.
The reference arm (--impl reference) times the CPU port of the reference (oracle/) on the box's
host cores on a bounded sample of the same workload and extrapolates by the reference's own
tile count (association.py:854-894).
--dump-outputs DIR writes what the last timed step computed (see dump_outputs); the inputs are
generated from fixed seeds, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (genes, cells, description)
    "coex_100k_x_20k": (20000, 100000, "large co-expression: 100k cells x 20k genes norm.coex (BASELINE configs[3], the "
                                       "size the metric is quoted on; fits one B200)"),
    "coex_10k_x_5k": (5000, 10000, "GSE123139-shaped: 10k cells x 5k genes norm.coex (BASELINE configs[1])"),
    "coex_2k_x_1k": (1000, 2000, "2,000 cells x 1,000 genes (BASELINE configs[0])"),
}
METRIC = "coex gene-pairs/s (r+P)"
UNIT = "pairs/s"
SEED = 1004
DUMP_SAMPLE = 1 << 19            # entries --dump-outputs keeps of a larger output
DUMP_BYTES = 64 << 20            # and the most it writes in all


def dump_outputs(path, arrays):
    """Write each array of ``arrays`` (name -> host or device array, None skipped) as <path>/<name>.npy
    in float64.  An array of more than DUMP_SAMPLE entries is written as the 1-D run of its entries at
    DUMP_SAMPLE positions drawn with a fixed seed (the same positions for every array of that shape),
    and the positions as <path>/<name>_index.npy: one row of coordinates per dimension."""
    import torch
    os.makedirs(path, exist_ok=True)
    files = {}
    for name, a in arrays.items():
        if a is None:
            continue
        t = torch.as_tensor(a)
        if t.numel() > DUMP_SAMPLE:
            flat = np.sort(np.random.default_rng(SEED).choice(t.numel(), DUMP_SAMPLE, replace=False, shuffle=False))
            files[name + "_index"] = np.array(np.unravel_index(flat, tuple(t.shape)), dtype=np.float64)
            t = t.reshape(-1)[torch.from_numpy(flat).to(t.device)]
        files[name] = t.to(torch.float64).cpu().numpy()
    total = sum(v.nbytes for v in files.values())
    assert total <= DUMP_BYTES, "--dump-outputs would write %d bytes" % total
    for name, v in files.items():
        np.save(os.path.join(path, name + ".npy"), v, allow_pickle=False)


def cpu_sample_genes(cores, n_gene):
    """Genes of the CPU sample: a whole number nb of the reference's 500-gene blocks, chosen so that
    its nb (nb + 1) / 2 tiles fill the thread pool's waves as evenly as possible (15 tiles on 16
    cores, 28 on 32): extrapolating by tile count then does not charge the CPU for idle threads."""
    best, best_eff = 4, 0.0
    for nb in range(4, 12):
        tiles = nb * (nb + 1) // 2
        eff = tiles / float(-(-tiles // cores) * cores)
        if eff > best_eff + 1e-9:
            best, best_eff = nb, eff
    return min(best * 500, n_gene)


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and throttle reasons of one GPU DURING the timed region: an NVML polling thread (20 ms; no
    start-up latency, so even a 100 ms region gets samples), nvidia-smi -lms as the fallback."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASON_BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.thread = None
        self.rows = []

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.gpu)

    def _poll(self, nv, h):
        import threading
        self.stop_flag = threading.Event()
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)

        def loop():
            while not self.stop_flag.is_set():
                try:
                    try:
                        bits = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), float(mx),
                                      nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(bits)))
                except Exception:
                    pass
                self.stop_flag.wait(0.02)
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def start(self):
        try:
            nv, h = self._nvml_handle()
            self._poll(nv, h)
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            if self.rows:
                pw = [r[2] for r in self.rows]
                load = [r[0] for r in self.rows if r[2] >= 0.5 * max(pw)] or [r[0] for r in self.rows]
                bits = 0
                for r in self.rows:
                    bits |= r[3]
                out.update(sm_mhz=float(np.median(load)), sm_max_mhz=float(max(r[1] for r in self.rows)),
                           reasons=sorted(k for k, b in self.REASON_BITS.items() if bits & b), samples=len(self.rows),
                           power_w_max=float(max(pw)), how="nvml, 20 ms")
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            # "under load": samples drawing more than half of the peak power seen
            load = [s for s, p_ in zip(sm, pw) if p_ >= 0.5 * max(pw)] or sm
            out.update(sm_mhz=float(np.median(load)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=float(max(pw)))
        return out


# --------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference)
# --------------------------------------------------------------------------------------
def reference_tiles(n_gene, bs=500):
    nb = (n_gene + bs - 1) // bs
    return nb * (nb + 1) // 2


def cpu_sample_problem(n_gene, n_cell):
    from normalisr_b200 import synth
    g = cpu_sample_genes(os.cpu_count() or 1, n_gene)
    p = synth.host_problem(SEED, g, n_cell, n_module=2, module_size=20)
    return p["dt"], p["dc"]


def cpu_time_once(dt, dc, setting):
    """One pass of the oracle over the sample.  setting 'A' = the reference CLI's configuration
    (BLAS pinned to one thread, bin/normalisr:3, thread pool over tiles with nth = all cores);
    'B' = nth=1 with BLAS using all cores."""
    import normalisr_oracle as orc
    cores = os.cpu_count()
    t0 = time.perf_counter()
    if setting == "A":
        try:
            from threadpoolctl import threadpool_limits
            with threadpool_limits(limits=1):
                orc.coex(dt, dc, nth=cores)
        except ImportError:
            orc.coex(dt, dc, nth=cores)
    else:
        orc.coex(dt, dc, nth=1)
    return time.perf_counter() - t0


def cpu_extrapolate(seconds, sample_genes, n_gene):
    """The reference executes reference_tiles(n_gene) tiles of <=500x500 genes; the sample is a
    whole number of such tiles, all over the full cell count, so time scales by the tile ratio."""
    per_tile = seconds / reference_tiles(sample_genes)
    total = per_tile * reference_tiles(n_gene)
    return (n_gene * (n_gene - 1) / 2) / total


def run_reference(args, n_gene, n_cell, wl_name, wl_desc):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dt, dc = cpu_sample_problem(n_gene, n_cell)
    sg = dt.shape[0]
    best = {}
    for setting in ("B", "A"):
        best[setting] = cpu_time_once(dt, dc, setting)          # also serves as warm-up
    setting = min(best, key=best.get)
    for _ in range(max(0, args.warmup - 1)):
        cpu_time_once(dt, dc, setting)
    ts = [cpu_time_once(dt, dc, setting) for _ in range(args.steps)]
    total = sum(ts)
    value = cpu_extrapolate(total / args.steps, sg, n_gene)
    sample = ("%d of %d genes x all %d cells = %d of the reference's %d 500x500 tiles per step (a tile count that fills "
              "the %d-thread pool's waves to %.0f %%), extrapolated by tile count; thread setting %s (%s); s per tile: "
              "A (BLAS=1 thread, nth=cores) %.3f, B (nth=1, BLAS=all cores) %.3f" % (
                  sg, n_gene, n_cell, reference_tiles(sg), reference_tiles(n_gene), os.cpu_count(),
                  100.0 * reference_tiles(sg) / (-(-reference_tiles(sg) // os.cpu_count()) * os.cpu_count()), setting,
                  "BLAS=1 thread, nth=cores" if setting == "A" else "nth=1, BLAS=all cores",
                  best["A"] / reference_tiles(sg), best["B"] / reference_tiles(sg)))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl_name, "genes": n_gene, "cells": n_cell, "covariates": int(dc.shape[0]), "note": wl_desc},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def run_ours(args, n_gene, n_cell, wl_name, wl_desc):
    import torch
    import torch.distributed as dist
    from normalisr_b200 import association, engine, parallel, synth
    from normalisr_b200 import normalisr as norm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = engine.context(local)
    if args.umma_pair is not None:
        engine.set_option("umma_pair", args.umma_pair)
    for kv in args.opt:
        k, v = kv.split("=")
        engine.set_option(k, int(v))
    precision = args.precision
    n_slices, n_products = engine.PRESETS[precision]

    # ---- synthetic inputs: this rank's block of genes, covariates identical on all ranks
    blk = parallel.row_split(n_gene, world)
    g0, g1 = rank * blk, min((rank + 1) * blk, n_gene)
    prob = synth.device_problem(SEED, g1 - g0, n_cell, dev, gene_seed=SEED * 1000 + rank)
    dt_dev, dc_dev = prob["dt"], prob["dc"]
    dc_np = dc_dev.cpu().numpy()
    pairs = n_gene * (n_gene - 1) / 2

    single = world == 1
    schedule = args.schedule
    if args.transport:
        parallel.TRANSPORT = args.transport
    if single:
        P = torch.empty((n_gene, n_gene), dtype=torch.float64, device=dev)
        D = torch.empty_like(P)
        tiles_full = engine.coex_tiles(n_gene)
        n_my_tiles = len(tiles_full)
        local_sl = engine.Sliced(n_gene, n_cell, n_slices, dev)
    else:
        if schedule == "pairs":
            my_rows = parallel.block_rows(n_gene, world, rank)
            n_my_tiles = int(parallel.owned_tile_mask(n_gene, world, rank).sum())
        else:
            t_tiles = (n_gene + 127) // 128
            a, b = parallel.strip_bounds(t_tiles, world)[rank]
            my_rows = min(b * 128, n_gene) - a * 128
            n_my_tiles = len(parallel.strip_tiles(t_tiles, a, b))
        P = torch.zeros((max(my_rows, 1), n_gene), dtype=torch.float64, device=dev)
        D = torch.zeros_like(P)
    contract_ms = []
    project_ms = []
    k_plan = {}

    def step_device(record=False):
        # the whole path, every step: covariate basis (Gram matrix + small factorisation), projection,
        # (block exchange,) contraction + P-values
        if not single:
            ev = [] if record else None
            pev = [] if record else None
            parallel.coex_sharded(dt_dev, dc_dev, n_gene, precision=precision, out=(P, D), schedule=schedule, events=ev,
                                  proj_events=pev)
            if record:
                contract_ms.append(ev)
                project_ms.extend(pev)
            return
        Qt_dev, crank, _ = association.covariate_basis_device(ctx, dc_dev)
        dof_a = (n_cell - 1 - crank) / 2
        if record:
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
        engine.residualize(ctx, dt_dev, Qt_dev, n_slices, out=local_sl, row_offset=0)
        if record:
            p1.record()
            project_ms.append((p0, p1))
        full = local_sl
        full.rows = n_gene
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if "k" not in k_plan:          # int32-overflow bound from the digit energies: planned once (tiny D2H)
            k_plan["k"] = engine.plan_k_chunk(full, full, n_products)
        engine.contract(ctx, engine.MODE_COEX, full, full, tiles_full, dof_a, P, D, n_products, k_chunk=k_plan["k"])
        if record:
            e1.record()
            contract_ms.append([(e0, e1)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing
    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = engine.LAUNCHES
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step_device(record=True)
    ev1.record()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = engine.LAUNCHES - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # what norm.coex returns: (P, dot, var)
        dump_outputs(args.dump_outputs, {"P": P, "dot": D, "var": local_sl.var})
    ms_step = ms_total / args.steps
    value = pairs / (ms_step * 1e-3)
    k_list = [sum(e0.elapsed_time(e1) for e0, e1 in evs) for evs in contract_ms]
    k_ms = float(np.mean(k_list)) if k_list else None
    # adaptive schedule (default preset, >= 8192 cells): 6 products on every tile + 8 on the refined ones
    refined, eff_products = None, float(n_products)
    if single and precision == "default" and any(kv.startswith("adaptive_min_cells=") and not kv.endswith("=0") for kv in args.opt):
        try:
            refined = engine.last_refined(ctx, n_my_tiles)
            eff_products = 6.0 + 8.0 * refined / n_my_tiles
        except Exception:
            refined = None

    # ---- the consumer of P (SURVEY 8f-1): per-row BH + threshold on the device-resident matrix
    binnet_info = None
    if single and not args.no_de:
        try:
            binnet_info = bench_binnet(torch, ctx, P, n_gene)
        except Exception as e:
            binnet_info = {"error": repr(e)[:300]}

    # ---- end to end through the public API, host buffers
    e2e = None
    if not args.no_e2e:
        dt_host = torch.empty((g1 - g0, n_cell), dtype=torch.float64, pin_memory=True)
        dt_host.copy_(dt_dev)
        if single:
            P_host = torch.empty((n_gene, n_gene), dtype=torch.float64, pin_memory=True)
            D_host = torch.empty((n_gene, n_gene), dtype=torch.float64, pin_memory=True)
        elif schedule == "pairs":
            # ONE (n_gene, n_gene) P and dot for the whole job, in a page-locked mapping shared by all ranks:
            # every GPU writes the rectangles it computed and their transposes, rank 0 holds the reference's
            # complete return value after the step's closing barrier
            (P_host, D_host), shared_home = parallel.shared_host_matrices(2, (n_gene, n_gene))
        else:
            P_host = torch.empty((max(my_rows, 1), n_gene), dtype=torch.float64, pin_memory=True)
            D_host = torch.empty((max(my_rows, 1), n_gene), dtype=torch.float64, pin_memory=True)
        del dt_dev, prob
        torch.cuda.empty_cache()

        def step_e2e():
            if single:
                norm.coex(dt_host, dc_np, precision=precision, out=(P_host, D_host))
            elif schedule == "pairs":
                parallel.coex_host(dt_host, dc_np, n_gene, precision=precision, out_dev=(P, D), home=(P_host, D_host))
            else:
                parallel.coex_host(dt_host, dc_np, n_gene, precision=precision, out_dev=(P, D), out_host=(P_host, D_host),
                                   schedule=schedule)

        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        for _ in range(min(args.warmup, 3)):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_e2e()
        barrier()
        sec = max_over_ranks(time.perf_counter() - t0)
        d2h_bytes = float(P_host.shape[0] * P_host.shape[1] * 16)
        if not single and schedule == "pairs":
            # this rank's diagonal block (both triangles) + every rectangle it computed and its transpose
            d2h_bytes = float(my_rows * my_rows * 16)
            for _, src, parity in parallel.exchange_plan(world, rank):
                a0, a1, b0, b1 = parallel._segment_rect(my_rows, parallel.block_rows(n_gene, world, src), parity)
                d2h_bytes += 2.0 * (a1 - a0) * (b1 - b0) * 16
        h2d_t = torch.tensor([float(dt_host.numel() * 8), d2h_bytes], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(h2d_t)
        e2e = {"value": pairs / (sec / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": int(h2d_t[0].item()),
               "d2h_bytes_per_step": int(h2d_t[1].item()), "steps": e2e_steps, "ms_per_step": 1e3 * sec / e2e_steps,
               "api": "normalisr_b200.normalisr.coex(dt_host, dc, out=pinned)" if single else
                      ("normalisr_b200.parallel.coex_host(dt_block_host, dc, n_gene, home=(P, dot)): one complete symmetric "
                       "P and dot for the job, both triangles, in a page-locked mapping %s" % (
                           "shared by all ranks (rank 0 holds the reference's return value)" if shared_home else
                           "per rank (/dev/shm too small for a shared one)") if schedule == "pairs" else
                       "normalisr_b200.parallel.coex_host(dt_block_host, dc, n_gene)")}

        # the same call as a user of the reference makes it: ordinary (pageable) numpy arrays in, fresh numpy
        # arrays out; informational, not the headline (the contract's e2e uses page-locked input)
        if single and e2e_steps >= 2 and not args.no_numpy_e2e:
            try:
                dt_np = np.empty(tuple(dt_host.shape), dtype=np.float64)
                dt_np[...] = dt_host.numpy()
                del P_host, D_host
                norm.coex(dt_np, dc_np, precision=precision)
                t0 = time.perf_counter()
                for _ in range(2):
                    res_np = norm.coex(dt_np, dc_np, precision=precision)
                sec_np = (time.perf_counter() - t0) / 2
                e2e["numpy_in_numpy_out"] = {"value": pairs / sec_np, "unit": UNIT, "ms_per_step": 1e3 * sec_np, "steps": 2,
                                             "api": "normalisr_b200.normalisr.coex(dt, dc) on pageable numpy arrays, fresh "
                                                    "numpy P / dot / var returned (staged through page-locked slots by a "
                                                    "host thread team)"}
                del res_np, dt_np
            except Exception as e:
                e2e["numpy_in_numpy_out"] = {"error": repr(e)[:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the tcgen05 contraction)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    my_pairs = n_my_tiles * 128 * 128.0          # ~unique pairs in this rank's tiles (each tile pair is computed once)
    alg_flops = 2.0 * n_cell * (pairs if single else my_pairs)
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(
            "%s/%s/%d" % (wl_name, precision, world))
    except Exception:
        pass
    roof = None
    if k_ms:
        ach = alg_flops / (k_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": traffic, "kernel": "contract_umma_kernel", "kernel_ms": k_ms,
                "kernel_ms_per_step": [round(x, 2) for x in k_list], "peak_source": peak_src,
                "executed_int8_tops": 2.0 * eff_products * n_my_tiles * 128 * 128 *
                                      engine.padded_cells(n_cell) / (k_ms * 1e-3) / 1e12,
                "digit_products_executed": eff_products, "tiles_refined": refined,
                "ceiling_frac": 2.0 / eff_products, "frac_of_ceiling": (ach / peak_tf) / (2.0 / eff_products),
                "note": "algorithmic flop = 2*cells per unique pair; the exact-integer kernel executes %.2f int8 digit-plane "
                        "products per pair at 2x the bf16 rate, so its ceiling on this scale is 2/%.2f of the bf16 peak (ceiling_frac); "
                        "frac_of_ceiling = how much of that the kernel reaches" % (eff_products, eff_products)}

    # ---- the box's dense int8 rate (cuBLASLt), the denominator of the EXECUTED tensor-pipe utilisation
    if roof is not None and single and not args.no_cpu:
        try:
            i8 = measure_int8_peak(torch, dev)
            roof["int8_peak"] = i8
            roof["executed_frac_of_int8_sustained"] = roof["executed_int8_tops"] / i8["int8_tops_sustained"]
            roof["executed_frac_of_int8_burst"] = roof["executed_int8_tops"] / i8["int8_tops_burst"]
        except Exception as e:
            roof["int8_peak"] = {"error": repr(e)[:200]}

    # ---- roofline of the projection (HBM-bound): algorithmic bytes per SURVEY 8(d) = 16 B per matrix element
    roof_proj = None
    if project_ms:
        pm = float(np.mean([a.elapsed_time(b) for a, b in project_ms]))
        hbm = peaks.get("hbm_gbs") or 6650.0
        elems = float(g1 - g0) * n_cell
        roof_proj = {"bound": "hbm", "achieved": 16.0 * elems / (pm * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                     "frac": 16.0 * elems / (pm * 1e-3) / 1e9 / hbm, "kernel": "coef_mma_kernel + residual_mma_kernel",
                     "kernel_ms": pm, "algorithmic_bytes": 16.0 * elems,
                     "executed_bytes": (16.0 + n_slices) * elems,
                     "executed_frac": (16.0 + n_slices) * elems / (pm * 1e-3) / 1e9 / hbm,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)",
                     "note": "algorithmic = 8 B read + 8 B residual written per element (SURVEY 8d); executed = X read "
                             "twice (coefficients, then residual + Hadamard + digits) + %d int8 digit planes written" % n_slices}

    # ---- CPU baseline on a bounded sample (N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        dt_s, dc_s = cpu_sample_problem(n_gene, n_cell)
        tb = {s: cpu_time_once(dt_s, dc_s, s) for s in ("B", "A")}
        s_best = min(tb, key=tb.get)
        cpu = {"value": cpu_extrapolate(tb[s_best], dt_s.shape[0], n_gene), "unit": UNIT, "cores": os.cpu_count(),
               "kind": "port",
               "sample": "%d of %d genes x all %d cells (%d of the reference's %d 500x500 tiles: fills the %d-thread pool's "
                         "waves to %.0f %%), one pass per thread setting, faster one (%s) extrapolated by tile count; "
                         "s per tile: A (BLAS=1 thread, nth=cores) %.3f, B (nth=1, BLAS=all cores) %.3f" % (
                             dt_s.shape[0], n_gene, n_cell, reference_tiles(dt_s.shape[0]), reference_tiles(n_gene),
                             os.cpu_count(), 100.0 * reference_tiles(dt_s.shape[0]) /
                             (-(-reference_tiles(dt_s.shape[0]) // os.cpu_count()) * os.cpu_count()), s_best,
                             tb["A"] / reference_tiles(dt_s.shape[0]), tb["B"] / reference_tiles(dt_s.shape[0]))}

    # ---- secondary metric of BASELINE.json: DE tests/s (config 3 shape), N = 1 only
    de = None
    normvar_info = None
    lcpm_info = None
    cvar_info = None
    if world == 1 and not args.no_de:
        try:
            de = bench_de(torch, dev, args)
        except Exception as e:          # the headline line must still be printed
            de = {"error": repr(e)[:300]}
        try:
            normvar_info = bench_normvar(torch, dev)
        except Exception as e:
            normvar_info = {"error": repr(e)[:300]}
        try:
            lcpm_info = bench_lcpm(torch, dev)
        except Exception as e:
            lcpm_info = {"error": repr(e)[:300]}
        try:
            cvar_info = bench_compute_var(torch, dev)
        except Exception as e:
            cvar_info = {"error": repr(e)[:300]}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": wl_name, "genes": n_gene, "cells": n_cell, "covariates": int(dc_np.shape[0]),
                   "precision": precision, "digit_planes": n_slices, "digit_products": n_products,
                   "cell_chunk": k_plan.get("k", 0),
                   "arithmetic": "f64 projection and epilogue; int8 x int8 -> int32 exact tensor-core sums",
                   "l2": "inputs (%.1f GB per rank) are larger than L2, no explicit flush" % ((g1 - g0) * n_cell * 8 / 1e9),
                   "parallelism": "1 GPU" if world == 1 else ("%d GPUs: gene-block projection, one all-gather of digit planes, tile-row strips" % world
                                   if schedule == "allgather" else
                                   "%d GPUs: gene-block projection, circulant block-pair schedule (%d point-to-point rounds "
                                   "of digit planes overlapped with the contraction, transport %s)" % (
                                       world, world // 2, "nccl" if (parallel.TRANSPORT == "nccl" or None in parallel._SYMM.values())
                                       else "copy engines over peer-mapped memory")),
                   "note": wl_desc},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "roofline_projection": roof_proj, "cpu_baseline": cpu,
        "de": de, "binnet": binnet_info, "normvar": normvar_info, "lcpm": lcpm_info, "compute_var": cvar_info,
    }
    if roof_proj is not None and k_ms:
        # rank 0's step on the device clock: projection, contraction (with N > 1 one persistent launch that starts on
        # the diagonal block while the exchange is in flight), and what is left: covariate basis, launch gaps, the
        # host-side planning between the two, exchange set-up and barriers
        line["timeline"] = {"step_ms": ms_step, "projection_ms": roof_proj["kernel_ms"], "contraction_ms": k_ms,
                            "other_ms": ms_step - roof_proj["kernel_ms"] - k_ms,
                            "rank": 0}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DE_WORKLOADS = {
    # name: (genes per GPU, cells, groupings, group_p, single, description)
    "de_50k_x_10k_x_300": (10000, 50000, 300, 0.02, 4,
                           "GSE120861-shaped CRISPRi screen DE: 50k cells x 10k genes x 300 gRNAs, norm.de(single=4): every gRNA "
                           "tested with the other 299 as covariates (BASELINE configs[2]); N > 1: 10k genes per GPU"),
    "de_1m_x_20k_x_1000": (2500, 1000000, 1000, 0.002, 0,
                           "atlas-scale DE sweep: 1M cells x 20k genes x 1,000 perturbations, gene blocks sharded over the GPUs "
                           "(BASELINE configs[4]); 2,500 genes per GPU"),
}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _de_cpu_sample(wl_name, seed):
    """Bounded CPU sample of a DE workload (host numpy, SURVEY 8d): returns (callable, scale, text);
    time(callable) * scale estimates the reference's time for ONE GPU's share of the workload."""
    import normalisr_oracle as orc
    from normalisr_b200 import synth
    genes, cells, groups, gp, single, _ = DE_WORKLOADS[wl_name]
    if single == 4:
        # the reference runs single=4 in y batches (association.py:866-875): one batch of genes x all cells x all gRNAs
        nc = 9
        bsy = orc._batch(0, 8, nc, cells, 500000)
        sg = min(genes, bsy)
        p = synth.host_problem(seed, sg, cells, n_group=groups, group_p=gp, n_module=0)
        n_batches = -(-genes // bsy)
        text = ("%d of %d genes (one of the reference's %d y-batches, association.py:866-875) x all %d cells x all %d gRNAs, "
                "oracle port de(single=4), time x %d" % (sg, genes, n_batches, cells, groups, n_batches))
        return (lambda: orc.de(p["dg"], p["dt"], p["dc"], single=4)), float(genes) / sg, text
    # single=0: the reference maps 500 x 500 tiles over (groupings, genes) at all cells; sample one tile at 1/16 of the cells
    sc = cells // 16
    p = synth.host_problem(seed, 500, sc, n_group=min(500, groups), group_p=max(gp, 0.002), n_module=0)
    tiles = (-(-groups // 500)) * (-(-genes // 500))
    text = ("one 500 x 500 tile of the reference's %d (groupings x genes) tiles at %d of %d cells, oracle port de(single=0), "
            "time x 16 x %d (SURVEY 8d: linear in cells and tiles)" % (tiles, sc, cells, tiles))
    return (lambda: orc.de(p["dg"], p["dt"], p["dc"])), 16.0 * tiles, text


def run_de_reference(args, wl_name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    genes, cells, groups, gp, single, desc = DE_WORKLOADS[wl_name]
    fn, scale, text = _de_cpu_sample(wl_name, SEED + 1)
    try:
        from threadpoolctl import threadpool_limits  # noqa: F401
    except ImportError:
        pass
    for _ in range(max(1, args.warmup)):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    sec = (time.perf_counter() - t0) / args.steps
    value = groups * genes / (sec * scale)                      # a rate: the same for every N under weak scaling
    line = {
        "impl": "reference", "metric": "DE tests/s (single=%d)" % single, "value": value, "unit": "tests/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl_name, "genes": genes * args.gpus, "cells": cells, "groupings": groups, "genes_per_gpu": genes,
                   "note": desc},
        "cpu_baseline": {"value": value, "unit": "tests/s", "cores": os.cpu_count(), "kind": "port",
                         "sample": text + "; nth=1, BLAS = all cores (the faster setting for this path in the survey)"},
        "e2e": {"value": value, "unit": "tests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def de_phase_times(torch, ctx, p, single, n_slices, n_products, reps=5, skip=2):
    """Device times of the phases of one de() call on device-resident inputs (CUDA events around the same
    engine calls the public API makes): covariate basis, projection of the groupings, projection of the
    genes, contraction(s), solve (single=4).  The first ``skip`` repetitions are not counted: their event
    brackets include the first device allocations of the outputs (the GPU idles while cudaMalloc runs)."""
    from normalisr_b200 import association, engine
    out = {}

    def timed(name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        out.setdefault(name, []).append((e0, e1))
        return r

    n = p["dt"].shape[1]
    for _ in range(reps):
        Qt, rank_c, _ = timed("basis", lambda: association.covariate_basis_device(ctx, p["dc"]))
        Rx, xd = timed("project_groupings", lambda: association._residualize_groupings(ctx, p["dg"], Qt, n_slices, single == 4))
        Ry = timed("project_genes", lambda: engine.residualize(ctx, p["dt"], Qt, n_slices))
        nx, ny = Rx.rows, Ry.rows
        if single == 0:
            P = torch.empty((nx, ny), dtype=torch.float64, device=ctx.device)
            G = torch.empty_like(P)
            timed("contract", lambda: engine.contract(ctx, engine.MODE_DE, Rx, Ry, engine.rect_tiles(nx, ny),
                                                     (n - 1 - rank_c) / 2, P, G, n_products))
        else:
            Gxy = torch.empty((nx, ny), dtype=torch.float64, device=ctx.device)
            Gxx = torch.empty((nx, nx), dtype=torch.float64, device=ctx.device)

            def grams():
                engine.contract(ctx, engine.MODE_RAW, Rx, Ry, engine.rect_tiles(nx, ny), 1.0, None, Gxy, n_products)
                if Rx.n_slices == 1:
                    engine.contract(ctx, engine.MODE_RAW, Rx, Rx, engine.rect_tiles(nx, nx), 1.0, None, Gxx, 1)
                    engine.gram_correct(ctx, Gxx, Rx.coef)
                    return Gxx
                return engine.gram_f64(ctx, xd, Rx.coef)
            g = timed("contract", grams)
            timed("solve", lambda: engine.de4_solve(ctx, g, Gxy, Ry.var * n, n, rank_c, 0, 1e-8, False))
    torch.cuda.synchronize()
    return {k: float(np.mean([a.elapsed_time(b) for a, b in v[skip:]])) for k, v in out.items()}, Rx.n_slices


def de_roofline(phases, planes_x, genes, cells, groups, single, n_slices, n_products):
    """Per-phase rooflines of one de() call from the phase times: projection of the genes (HBM,
    algorithmic 16 B per element, SURVEY 8d), contraction (tensor, 2 n flop per test + the groupings'
    Gram matrix for single=4), solve."""
    peaks = _peaks()
    hbm = peaks.get("hbm_gbs") or 6650.0
    tf = peaks.get("bf16_tflops_sustained") or 1400.0
    src = "of measured" if peaks else "of fallback"
    proj_ms = phases["project_genes"]
    alg_proj = 16.0 * genes * cells
    con_ms = phases["contract"]
    flop = 2.0 * cells * groups * genes + (2.0 * cells * groups * (groups + 1) / 2 if single == 4 else 0.0)
    prods = n_slices if planes_x == 1 else n_products
    roof_phases = {
        "project_genes": {"bound": "hbm", "ms": proj_ms, "achieved": alg_proj / (proj_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                          "frac": alg_proj / (proj_ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes": alg_proj,
                          "executed_bytes": (16.0 + n_slices) * genes * cells},
        "project_groupings": {"bound": "hbm", "ms": phases["project_groupings"],
                              "achieved": 16.0 * groups * cells / (phases["project_groupings"] * 1e-3) / 1e9, "peak": hbm,
                              "unit": "GB/s", "frac": 16.0 * groups * cells / (phases["project_groupings"] * 1e-3) / 1e9 / hbm,
                              "digit_planes": planes_x},
        "contract": {"bound": "tensor", "ms": con_ms, "achieved": flop / (con_ms * 1e-3) / 1e12, "peak": tf, "unit": "TFLOP/s",
                     "frac": flop / (con_ms * 1e-3) / 1e12 / tf, "algorithmic_flop": flop,
                     "digit_products_executed": prods, "ceiling_frac": 2.0 / prods},
    }
    if "solve" in phases:
        roof_phases["solve"] = {"bound": "latency", "ms": phases["solve"],
                                "note": "blocked Cholesky of the %d x %d Gram matrix + w = K Gxy + closed form + P-values" % (groups, groups)}
    dom = max(("project_genes", "contract"), key=lambda k: roof_phases[k]["ms"])
    return dict(roof_phases[dom], kernel=("coef_mma_kernel + residual_mma_kernel" if dom == "project_genes" else "contract_umma_kernel"),
                kernel_ms=roof_phases[dom]["ms"], traffic=None, peak_source="MEASURED_PEAKS.json (%s)" % src, phases=roof_phases,
                phase_ms={k: round(v, 3) for k, v in phases.items()})


def de_cpu_baseline(wl_name):
    genes, cells, groups, gp, single, _ = DE_WORKLOADS[wl_name]
    fn, scale, text = _de_cpu_sample(wl_name, SEED + 1)
    t0 = time.perf_counter()
    fn()
    sec = time.perf_counter() - t0
    return {"value": groups * genes / (sec * scale), "unit": "tests/s", "cores": os.cpu_count(), "kind": "port",
            "sample": text + "; nth=1, BLAS = all cores; one timed pass (%.1f s)" % sec}


def run_de(args, wl_name):
    """DE tests/s through the public API norm.de, genes sharded over ranks with no exchange step
    (weak scaling: a fixed gene block per GPU)."""
    import torch
    import torch.distributed as dist
    from normalisr_b200 import engine, synth
    from normalisr_b200 import normalisr as norm
    genes, cells, groups, gp, single, desc = DE_WORKLOADS[wl_name]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = engine.context(local)
    precision = args.precision
    n_slices, n_products = engine.PRESETS[precision]
    p = synth.device_problem(SEED + 1, genes, cells, dev, n_group=groups, group_p=gp, gene_seed=SEED * 77 + rank, n_module=0)
    total_genes = genes * world
    tests = float(groups) * total_genes

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step():
        return norm.de(p["dg"], p["dt"], p["dc"], single=single, precision=precision)

    # each step's result stays alive while the next one runs, in the warm-up too, so that the timed steps
    # find the allocator's cache already sized for two results
    for _ in range(args.warmup):
        res = step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = engine.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    barrier()
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = engine.LAUNCHES - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("P", "gamma", "alpha", "varg", "vart"), res)))
    del res
    phases, planes_x = de_phase_times(torch, ctx, p, single, n_slices, n_products)

    # ---- end to end: pinned host dg / dt / dc in, host P / gamma / variances out
    e2e = None
    if not args.no_e2e:
        try:
            hosts = {k: torch.empty(p[k].shape, dtype=torch.float64, pin_memory=True).copy_(p[k]) for k in ("dg", "dt", "dc")}
            torch.cuda.synchronize()
            del p
            torch.cuda.empty_cache()
            steps_e = max(1, min(args.steps, args.e2e_steps))
            for _ in range(min(args.warmup, 2)):
                res = norm.de(hosts["dg"], hosts["dt"], hosts["dc"], single=single, precision=precision)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps_e):
                res = norm.de(hosts["dg"], hosts["dt"], hosts["dc"], single=single, precision=precision)
            barrier()
            sec = max_over_ranks(time.perf_counter() - t0) / steps_e
            h2d = sum(v.numel() * 8 for v in hosts.values()) * world
            d2h = sum(r.nbytes for r in res if r is not None) * world
            e2e = {"value": tests / sec, "unit": "tests/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                   "steps": steps_e, "ms_per_step": 1e3 * sec, "api": "normalisr_b200.normalisr.de(dg_host, dt_host, dc_host, single=%d)" % single}
        except Exception as e:
            e2e = {"error": repr(e)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    roof = de_roofline(phases, planes_x, genes, cells, groups, single, n_slices, n_products)
    cpu = de_cpu_baseline(wl_name) if (world == 1 and not args.no_cpu) else None
    line = {
        "metric": "DE tests/s (single=%d)" % single, "value": tests / (ms_step * 1e-3), "unit": "tests/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl_name, "genes": total_genes, "cells": cells, "groupings": groups, "genes_per_gpu": genes,
                   "single": single, "precision": precision, "grouping_planes": planes_x,
                   "arithmetic": "f64 projection, solve and epilogue; int8 x int8 -> int32 exact tensor-core sums",
                   "l2": "inputs (%.1f GB per rank) are larger than L2, no explicit flush" % (genes * cells * 8 / 1e9),
                   "parallelism": "1 GPU" if world == 1 else "%d GPUs: gene blocks, no exchange" % world, "note": desc},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_int8_peak(torch, dev, seconds=3.0):
    """Dense int8 tensor-core throughput of this box (cuBLASLt through torch._int_mm, 8192^3): best of
    10 (burst) and back to back for ``seconds`` (sustained, under the power cap) - the denominator of
    the contraction's EXECUTED int8 utilisation.  Library call, measurement only."""
    n = 8192
    a = torch.randint(-128, 127, (n, n), dtype=torch.int8, device=dev)
    b = torch.randint(-128, 127, (n, n), dtype=torch.int8, device=dev)
    for _ in range(3):
        torch._int_mm(a, b)
    torch.cuda.synchronize()
    ops = 2.0 * n ** 3
    best = 0.0
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch._int_mm(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, ops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(20, int(seconds / (ops / (best * 1e12))))
    e0.record()
    for _ in range(reps):
        torch._int_mm(a, b)
    e1.record()
    torch.cuda.synchronize()
    sus = reps * ops / (e0.elapsed_time(e1) * 1e-3) / 1e12
    return {"int8_tops_burst": best, "int8_tops_sustained": sus, "how": "torch._int_mm 8192^3, best of 10 / %d back to back" % reps}


def bench_binnet(torch, ctx, P, n_gene, qcut=0.05, reps=5):
    """normalisr_b200.binnet on the (n_gene, n_gene) P left on the device by coex: HBM-bound,
    9 B per entry (8 read + 1 written)."""
    from normalisr_b200 import binnet as bn
    out = torch.empty((n_gene, n_gene), dtype=torch.uint8, device=P.device)
    stats = torch.zeros(2, dtype=torch.int64, device=P.device)
    for _ in range(2):
        bn.binnet_rows(ctx, P, qcut, 0, out=out, stats=stats)
    stats.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        bn.binnet_rows(ctx, P, qcut, 0, out=out, stats=stats)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    edges = int(stats[0].item()) // reps
    # the same rows through the first-generation kernel (8-byte row staged per SM with one bulk copy), for comparison
    from normalisr_b200 import engine as _engine
    _engine.set_option("binnet_keys", 0)
    try:
        bn.binnet_rows(ctx, P, qcut, 0, out=out, stats=stats)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            bn.binnet_rows(ctx, P, qcut, 0, out=out, stats=stats)
        e1.record()
        torch.cuda.synchronize()
        ms_values = e0.elapsed_time(e1) / reps
    finally:
        _engine.set_option("binnet_keys", 1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs") or peaks.get("hbm_GBs") or 6545.0
    gbs = 9.0 * n_gene * n_gene / (ms * 1e-3) / 1e9
    return {"workload": "binnet_%dk" % (n_gene // 1000), "qcut": qcut, "ms": ms, "ms_values_kernel": ms_values, "edges": edges,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes": 9 * n_gene * n_gene}}


def bench_normvar(torch, dev, n_gene=10000, n_cell=50000, reps=3):
    """normalisr_b200.normvar (the step upstream of coex / de) on device-resident inputs: 16 B of
    algorithmic traffic per matrix entry (8 read + 8 written); the kernels read dt twice and spend
    one float64 exp per entry in each pass."""
    from normalisr_b200 import normalisr as norm, synth
    torch.cuda.empty_cache()
    p = synth.device_problem(1002, n_gene, n_cell, dev)
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    w = torch.exp(0.3 * torch.randn(n_cell, generator=g, device=dev, dtype=torch.float64))
    wt = torch.rand(n_gene, generator=g, device=dev, dtype=torch.float64) * 1.5
    for _ in range(2):
        norm.normvar(p["dt"], p["dc"], w, wt)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        norm.normvar(p["dt"], p["dc"], w, wt)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs") or 6545.0
    gbs = 16.0 * n_gene * n_cell / (ms * 1e-3) / 1e9
    del p
    torch.cuda.empty_cache()
    return {"workload": "normvar_%dk_x_%dk" % (n_cell // 1000, n_gene // 1000), "covariates": 9, "ms": ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes": 16 * n_gene * n_cell,
                         "note": "two passes over dt; the statistics pass is a skinny float64 tensor-core GEMM with one exp per entry"}}


def bench_lcpm(torch, dev, n_gene=10000, n_cell=50000, reps=3):
    """normalisr_b200.lcpm on a device-resident int32 count matrix: 12 B of algorithmic traffic per
    entry (4 read + 8 written); the kernels read the counts twice."""
    from normalisr_b200 import normalisr as norm
    torch.cuda.empty_cache()
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    lam = torch.rand((n_gene, 1), generator=g, device=dev) ** 3 * 20 + 0.05
    reads = torch.poisson(lam.expand(n_gene, n_cell), generator=g).to(torch.int32)
    reads[0] += 1
    for _ in range(2):
        norm.lcpm(reads)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        norm.lcpm(reads)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs") or 6545.0
    gbs = 12.0 * n_gene * n_cell / (ms * 1e-3) / 1e9
    del reads
    torch.cuda.empty_cache()
    return {"workload": "lcpm_%dk_x_%dk" % (n_cell // 1000, n_gene // 1000), "ms": ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes": 12 * n_gene * n_cell}}


def bench_compute_var(torch, dev, n_gene=10000, n_cell=50000, reps=3):
    """normalisr_b200.compute_var on device-resident inputs: 8 B of algorithmic traffic per entry
    (dt read once); the kernels read dt twice (coefficients / moments, then the column pass)."""
    from normalisr_b200 import normalisr as norm, synth
    torch.cuda.empty_cache()
    p = synth.device_problem(1002, n_gene, n_cell, dev)
    for _ in range(2):
        norm.compute_var(p["dt"], p["dc"])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        norm.compute_var(p["dt"], p["dc"])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs") or 6545.0
    gbs = 8.0 * n_gene * n_cell / (ms * 1e-3) / 1e9
    del p
    torch.cuda.empty_cache()
    return {"workload": "compute_var_%dk_x_%dk" % (n_cell // 1000, n_gene // 1000), "covariates": 9, "ms": ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes": 8 * n_gene * n_cell}}


def bench_de(torch, dev, args, n_gene=10000, n_cell=50000, n_group=300):
    """DE tests/s on the GSE120861-shaped config (BASELINE configs[2]: 50k cells x 10k genes x 300 gRNAs)
    through the public API: single=4 ("untested gRNAs as covariates", the configuration BASELINE names)
    with its per-phase roofline, a CPU baseline on a bounded sample and an end-to-end number from
    pinned host buffers; single=0 and single=1 device-resident times beside it."""
    from normalisr_b200 import engine, normalisr as norm, synth
    torch.cuda.empty_cache()
    ctx = engine.context(dev.index)
    n_slices, n_products = engine.PRESETS["default"]
    p = synth.device_problem(1003, n_gene, n_cell, dev, n_group=n_group, group_p=0.02)
    out = {"workload": "de_50k_x_10k_x_300", "genes": n_gene, "cells": n_cell, "groupings": n_group, "unit": "tests/s",
           "metric": "DE tests/s"}
    for single in (0, 4):
        for _ in range(3):
            norm.de(p["dg"], p["dt"], p["dc"], single=single)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps):
            norm.de(p["dg"], p["dt"], p["dc"], single=single)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out["single%d" % single] = {"value": n_group * n_gene / (ms * 1e-3), "ms": ms}
    phases, planes_x = de_phase_times(torch, ctx, p, 4, n_slices, n_products)
    out["value"] = out["single4"]["value"]
    out["ms_per_step"] = out["single4"]["ms"]
    out["roofline"] = de_roofline(phases, planes_x, n_gene, n_cell, n_group, 4, n_slices, n_products)
    # low-MOI design for single=1: 45 % of the cells carry no gRNA, the others one (a few two)
    g = torch.Generator(device=dev)
    g.manual_seed(1004)
    u = torch.rand(n_cell, generator=g, device=dev)
    who = torch.randint(0, n_group, (2, n_cell), generator=g, device=dev)
    dg1 = torch.zeros((n_group, n_cell), dtype=torch.float64, device=dev)
    one = torch.nonzero(u >= 0.45).squeeze(1)
    dg1[who[0, one], one] = 1
    two = torch.nonzero(u >= 0.95).squeeze(1)
    dg1[who[1, two], two] = 1
    for _ in range(2):
        norm.de(dg1, p["dt"], p["dc"], single=1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        norm.de(dg1, p["dt"], p["dc"], single=1)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    out["single1"] = {"value": n_group * n_gene / (ms * 1e-3), "ms": ms, "design": "low MOI: 45% of cells without gRNA"}
    del dg1
    # end to end (single=4): pinned host dg / dt / dc in, host outputs back
    if not args.no_e2e:
        try:
            hosts = {k: torch.empty(p[k].shape, dtype=torch.float64, pin_memory=True).copy_(p[k]) for k in ("dg", "dt", "dc")}
            torch.cuda.synchronize()
            for _ in range(2):
                res = norm.de(hosts["dg"], hosts["dt"], hosts["dc"], single=4)
            t0 = time.perf_counter()
            for _ in range(3):
                res = norm.de(hosts["dg"], hosts["dt"], hosts["dc"], single=4)
            sec = (time.perf_counter() - t0) / 3
            out["e2e"] = {"value": n_group * n_gene / sec, "unit": "tests/s", "ms_per_step": 1e3 * sec,
                          "h2d_bytes_per_step": int(sum(v.numel() * 8 for v in hosts.values())),
                          "d2h_bytes_per_step": int(sum(r.nbytes for r in res if r is not None)),
                          "api": "normalisr_b200.normalisr.de(dg_host, dt_host, dc_host, single=4)"}
            del hosts
        except Exception as e:
            out["e2e"] = {"error": repr(e)[:300]}
    del p
    torch.cuda.empty_cache()
    if not args.no_cpu:
        try:
            out["cpu_baseline"] = de_cpu_baseline("de_50k_x_10k_x_300")
        except Exception as e:
            out["cpu_baseline"] = {"error": repr(e)[:300]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="coex_100k_x_20k", choices=sorted(WORKLOADS) + sorted(DE_WORKLOADS))
    ap.add_argument("--precision", default="default", choices=["fast", "default", "precise"])
    ap.add_argument("--e2e-steps", type=int, default=1000000, help="cap on the e2e steps (default: same as --steps)")
    ap.add_argument("--schedule", default="pairs", choices=["pairs", "allgather"],
                    help="multi-GPU exchange schedule (normalisr_b200.parallel)")
    ap.add_argument("--transport", default=None, choices=["nccl", "ce", "auto"],
                    help="multi-GPU plane exchange: NCCL send/recv or copy-engine pulls from peer-mapped memory")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numpy-e2e", action="store_true", help="skip the informational pageable-numpy end-to-end call")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-de", action="store_true", help="skip the secondary DE tests/s measurement")
    ap.add_argument("--umma-pair", type=int, default=None, help="test hook: 1 = cta_group::2 kernel, 0 = single-CTA")
    ap.add_argument("--opt", action="append", default=[], help="test hook: name=value for nsr_set_option")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays the last one computed as DIR/<name>.npy (float64; "
                         "an array of more than %d entries as a fixed, seeded sample of its entries)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs takes --impl ours on one GPU")
    if args.workload in DE_WORKLOADS:
        if args.impl == "reference":
            run_de_reference(args, args.workload)
        else:
            run_de(args, args.workload)
        return
    n_gene, n_cell, desc = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, n_gene, n_cell, args.workload, desc)
    else:
        run_ours(args, n_gene, n_cell, args.workload, desc)


if __name__ == "__main__":
    main()
