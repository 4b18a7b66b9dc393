#!/usr/bin/env python3
"""Every gene's k strongest partners (norm.coextop) against the ways to get them without it.

  100,000 cells x 20,000 genes (bench.py's recipe and seed), k = 50:
    device input  coextop on device tensors            against  coex on device tensors (P and dot on the device)
    numpy input   coextop on numpy arrays (numpy out)  against  coex on numpy arrays, then a host top-k of
                                                                every row of r2 = dot^2 / (var_i var_j)
  and the split of coextop's device time between the contraction and the selection kernels (CUDA events
  around every strip's two launches, in a run of its own);
  150,000 genes x 4,096 cells, k = 50, device input: a run that coex cannot do on one GPU (P + dot: 360 GB).

Host clock around whole calls that end with their results where the caller wants them (a device synchronise
for device results), arms alternated after one warm-up call of each; peak device memory from torch's allocator
above what was allocated before the call.  The results of coextop are compared with the host top-k of coex's
P, dot and var.  The card's name and power limit are read in the same run and recorded beside the numbers.
python tools/coextop_bench.py --out profiles/coextop_b200.json

With ``--devices all`` (or a list such as ``0,1``) the run measures the several-GPU path instead:
  numpy input at 100,000 cells x 20,000 genes and at 150,000 genes x 4,096 cells, k = 50: coextop on one GPU
  against parallel.coextop_all_devices (the team path, also with a single device), arms alternated after one
  warm-up call of each, results compared bit for bit,
  and the digit-plane bytes each GPU pulls from its peers (from the shapes and the dealing, not timed);
  the merge kernel alone (nsr_topk_merge, CUDA events over --merge-reps launches): 8 parts of 18,750 rows with
  k = 50 (one owner's share at 150,000 genes on 8 GPUs, 240 MB of slots: more than the L2) and 8 parts of 2,000
  rows with k = 2,048.
python tools/coextop_bench.py --devices all --out profiles/coextop_devices_b200.json"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SEED = 1004        # bench.py's


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count(),
            "nvidia_smi": (q.stdout.strip() or q.stderr.strip()).splitlines()}


def timed(fn):
    """(seconds, peak device bytes above the allocation before the call, result)."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    return dt, torch.cuda.max_memory_allocated() - base, res


def host_topk(P, D, var, k, block=512):
    """Exact host top-k of r2 per row (key descending, column ascending), diagonal excluded: argpartition for
    k + 64 candidates, lexsort among them; a row whose boundary is tied beyond that margin is sorted whole."""
    G = D.shape[0]
    idx = np.empty((G, k), dtype=np.int64)
    cols = np.arange(G)
    m = min(G - 1, k + 64)
    for a in range(0, G, block):
        b = min(a + block, G)
        key = D[a:b] * D[a:b] / (var[a:b, None] * var[None, :])
        key[np.arange(b - a), np.arange(a, b)] = -1.0
        cand = np.argpartition(-key, m - 1, axis=1)[:, :m]
        for r in range(b - a):
            c = cand[r]
            kc = key[r, c]
            o = np.lexsort((c, -kc))
            if m < G - 1 and kc[o[-1]] >= kc[o[k - 1]]:
                o = np.lexsort((cols, -key[r]))
                idx[a + r] = cols[o[:k]]
            else:
                idx[a + r] = c[o[:k]]
    rows = np.arange(G)[:, None]
    return idx, P[rows, idx], D[rows, idx]


def same(got, want):
    return all(np.array_equal(np.asarray(g).view(np.int64), np.asarray(w).view(np.int64)) for g, w in zip(got, want))


def kernel_split(dt, dc, k):
    """ms of the contraction launches and of the selection launches inside one coextop call (CUDA events)."""
    from normalisr_b200 import coex as cx, engine
    from normalisr_b200 import normalisr as norm
    evs = {"contract": [], "select": []}
    real = {"contract": engine.contract, "select": engine.topk_strip}

    def wrap(name):
        def f(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            real[name](*a, **kw)
            e1.record()
            evs[name].append((e0, e1))
        return f

    engine.contract, engine.topk_strip = wrap("contract"), wrap("select")
    try:
        norm.coextop(dt, dc, k)
        torch.cuda.synchronize()
    finally:
        engine.contract, engine.topk_strip = real["contract"], real["select"]
    out = {name: sum(a.elapsed_time(b) for a, b in v) for name, v in evs.items()}
    out["strips"] = len(evs["select"])
    out["strip_rows"] = min(cx._STRIP_BYTES // (16 * 128 * dt.shape[0]) * 128, dt.shape[0])
    out["select_over_contract"] = out["select"] / out["contract"]
    return out


def merge_kernel(n_parts, rows, k, reps):
    """ms per nsr_topk_merge launch over ``reps`` back-to-back launches (CUDA events) on ``n_parts`` parts of
    ``rows`` x k filled slots with random keys (columns disjoint across parts); the result is checked once
    against a sort of the union."""
    from normalisr_b200 import engine
    ctx = engine.context(0)
    g = torch.Generator(device="cuda").manual_seed(SEED)
    parts, keys, cols = [], [], []
    for q in range(n_parts):
        key = torch.rand((rows, k), dtype=torch.float64, device="cuda", generator=g).sort(dim=1, descending=True)[0]
        col = q + n_parts * torch.arange(k, device="cuda").expand(rows, k)
        st = torch.empty((rows, k, 4), dtype=torch.float64, device="cuda")
        st[..., 0], st[..., 1], st[..., 2] = key, -key, 2 * key
        st.view(torch.int32).view(rows, k, 8)[..., 6:] = torch.stack([col, torch.zeros_like(col)], -1).to(torch.int32)
        parts.append(st)
        keys.append(key)
        cols.append(col)
    key, col = torch.cat(keys, 1), torch.cat(cols, 1)
    o = torch.sort(col, dim=1, stable=True)[1]
    o = o.gather(1, torch.sort(key.gather(1, o), dim=1, descending=True, stable=True)[1])[:, :k]
    idx, P_k, dot_k = engine.topk_merge(ctx, parts)
    ok = bool(torch.equal(idx, col.gather(1, o)) and torch.equal(P_k, -key.gather(1, o)) and
              torch.equal(dot_k, 2 * key.gather(1, o)))
    ptrs = (ctypes.c_void_p * n_parts)(*[t.data_ptr() for t in parts])
    status = torch.zeros(1, dtype=torch.int32, device="cuda")

    def launch():
        engine._lib.check(ctx.lib.nsr_topk_merge(ctx.handle, torch.cuda.current_stream().cuda_stream, ptrs, n_parts,
                                                 rows, k, idx.data_ptr(), P_k.data_ptr(), dot_k.data_ptr(),
                                                 status.data_ptr()), "nsr_topk_merge")
    for _ in range(10):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = n_parts * rows * k * 32 + rows * k * 24
    return {"parts": n_parts, "rows": rows, "k": k, "launches": reps, "ms_per_launch": ms,
            "slot_bytes_read": n_parts * rows * k * 32, "output_bytes": rows * k * 24,
            "GBps_on_those_bytes": nbytes / ms / 1e6, "identical_to_sort": ok and int(status.item()) == 0}


def devices_run(args, res):
    """One GPU against ``args.devices`` from numpy input at both shapes, and the merge kernel alone."""
    from normalisr_b200 import engine, parallel, synth
    from normalisr_b200 import normalisr as norm
    devs = parallel.visible_devices(args.devices if args.devices == "all" else
                                    [int(d) for d in args.devices.split(",")])
    res["devices"] = [str(d) for d in devs]
    k = args.k
    res["merge_kernel"] = [merge_kernel(8, 18750, 50, args.merge_reps), merge_kernel(8, 2000, 2048, args.merge_reps)]
    print(json.dumps({"merge_kernel": res["merge_kernel"]}), flush=True)
    res["arms"] = []
    for genes, cells in ((args.genes, args.cells), (args.big_genes, args.big_cells)):
        p = synth.device_problem(SEED, genes, cells, "cuda")
        dt_h, dc_h = p["dt"].cpu().numpy(), p["dc"].cpu().numpy()
        del p
        torch.cuda.empty_cache()
        # the team path itself (coextop(devices=) sends a one-device list down the one-GPU path)
        arms = {"one_gpu": lambda: norm.coextop(dt_h, dc_h, k),
                "all_devices": lambda: parallel.coextop_all_devices(dt_h, dc_h, k, devices=devs)}
        outs = {name: fn() for name, fn in arms.items()}
        times = {name: [] for name in arms}
        for _ in range(args.reps):
            for name, fn in arms.items():
                t = time.perf_counter()
                fn()
                times[name].append(time.perf_counter() - t)
        deal = parallel.coextop_deal(genes, len(devs))
        plane_bytes = engine.Sliced.storage_bytes(1, cells, engine.PRESETS["default"][0]) - \
            engine.Sliced.storage_bytes(0, cells, engine.PRESETS["default"][0])
        arm = {"genes": genes, "cells": cells, "k": k, "world": len(devs),
               "s": times, "median_s": {name: float(np.median(v)) for name, v in times.items()},
               "identical": same(outs["all_devices"], outs["one_gpu"]),
               "pulled_plane_bytes_per_gpu_not_timed": [sum((deal[s].hi - deal[s].lo) * plane_bytes for s in d.pulls)
                                                        for d in deal]}
        res["arms"].append(arm)
        print(json.dumps(arm), flush=True)
        del outs, dt_h, dc_h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--genes", type=int, default=20000)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big-genes", type=int, default=150000)
    ap.add_argument("--big-cells", type=int, default=4096)
    ap.add_argument("--devices", default=None, help='"all" or a list like 0,1: the several-GPU runs instead')
    ap.add_argument("--merge-reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from normalisr_b200 import normalisr as norm, synth
    torch.cuda.set_device(0)
    res = {"card": card(), "shape": {"cells": args.cells, "genes": args.genes, "k": args.k}, "reps": args.reps}
    if args.devices:
        devices_run(args, res)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
        print(json.dumps(res))
        return
    p = synth.device_problem(SEED, args.genes, args.cells, "cuda")
    dt_d, dc_d = p["dt"], p["dc"]
    dt_h, dc_h = dt_d.cpu().numpy(), dc_d.cpu().numpy()
    k = args.k

    # device input
    arms = {"coextop": lambda: norm.coextop(dt_d, dc_d, k), "coex": lambda: norm.coex(dt_d, dc_d)}
    dev = {name: [] for name in arms}
    for name, fn in arms.items():
        fn()
    for _ in range(args.reps):
        for name, fn in arms.items():
            t, peak, out = timed(fn)
            dev[name].append((t, peak))
            del out
    res["device_input"] = {name: {"s": [t for t, _ in v], "median_s": float(np.median([t for t, _ in v])),
                                  "peak_device_bytes": max(pk for _, pk in v)} for name, v in dev.items()}
    torch.cuda.empty_cache()
    res["kernel_split_ms"] = kernel_split(dt_d, dc_d, k)

    # numpy input: coextop against coex + host top-k
    host = {"coextop": [], "coex": [], "host_topk": []}
    norm.coextop(dt_h, dc_h, k)
    norm.coex(dt_h, dc_h)
    for _ in range(args.reps):
        t, peak, top = timed(lambda: norm.coextop(dt_h, dc_h, k))
        host["coextop"].append((t, peak))
        t, peak, cx = timed(lambda: norm.coex(dt_h, dc_h))
        host["coex"].append((t, peak))
        t0 = time.perf_counter()
        ref = host_topk(cx[0], cx[1], cx[2], k)
        host["host_topk"].append((time.perf_counter() - t0, 0))
        del cx
    res["numpy_input"] = {name: {"s": [t for t, _ in v], "median_s": float(np.median([t for t, _ in v])),
                                 "peak_device_bytes": max(pk for _, pk in v)} for name, v in host.items()}
    res["numpy_input"]["coex_plus_host_topk_median_s"] = (res["numpy_input"]["coex"]["median_s"] +
                                                         res["numpy_input"]["host_topk"]["median_s"])
    res["numpy_input"]["identical_to_host_topk"] = same(top[:3], ref)
    print(json.dumps({"device_input": res["device_input"], "kernel_split_ms": res["kernel_split_ms"],
                      "numpy_input": res["numpy_input"]}), flush=True)
    del p, dt_d, dc_d, dt_h, top, ref
    torch.cuda.empty_cache()

    # beyond coex on one GPU
    if args.big_genes:
        q = synth.device_problem(SEED, args.big_genes, args.big_cells, "cuda")
        norm.coextop(q["dt"][:2000], q["dc"], k)
        t, peak, out = timed(lambda: norm.coextop(q["dt"], q["dc"], k))
        idx = out[0]
        ok = bool((idx != torch.arange(idx.shape[0], device=idx.device)[:, None]).all())
        split = kernel_split(q["dt"], q["dc"], k)
        res["big"] = {"genes": args.big_genes, "cells": args.big_cells, "k": k, "s": t, "peak_device_bytes": peak,
                      "input_bytes": q["dt"].numel() * 8, "coex_P_dot_bytes": 16 * args.big_genes ** 2,
                      "no_self_partner": ok, "kernel_split_ms": split}
        print(json.dumps({"big": res["big"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
