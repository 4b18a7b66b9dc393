#!/usr/bin/env python3
"""lcpm on sparse counts against the dense path, on one GPU (default 50,000 cells x 10,000 genes at densities 0.05,
0.10 and 0.30; counts drawn on the device from a fixed seed):

  device   norm.lcpm on a CUDA int32 matrix against the same counts as a CUDA CSR tensor (int64 row pointers, int32
           cell indices and counts).  CUDA events around whole calls, after warm-up; the inputs are larger than the
           126 MB L2 at every density.  GB/s on algorithmic bytes: the counts read by both passes (4 B per entry
           dense; 8 B per stored entry + 8 B per row pointer as CSR) + 8 B per output entry written.
  e2e      from a scipy CSR matrix with numpy out: norm.lcpm(csr) against what the previous release did with it,
           norm.lcpm(csr.toarray()) (the host densification included); host clock, both arms alternated.
           The outputs of the two arms are compared bit for bit in the same run, as are the device arms.

The card's name and power limit are recorded beside the numbers.
python tools/lcpm_sparse_bench.py --out profiles/lcpm_sparse_b200.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def counts(genes, cells, density, seed):
    """(genes x cells) int32 counts on the device: an entry is stored with probability `density`, stored counts are
    1 + geometric (mean ~3), the first gene is non-zero in every cell (no empty cell)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((genes, cells), dtype=torch.int32, device="cuda")
    step = max(1, (1 << 28) // (4 * cells))
    for g0 in range(0, genes, step):
        g1 = min(genes, g0 + step)
        u = torch.rand((g1 - g0, cells), generator=g, device="cuda")
        c = 1 + torch.floor(-torch.log(torch.rand((g1 - g0, cells), generator=g, device="cuda")) * 2.5)
        out[g0:g1] = torch.where(u < density, c, torch.zeros_like(c)).to(torch.int32)
    out[0].clamp_(min=1)
    return out


def time_device(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return ts


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--genes", type=int, default=10000)
    ap.add_argument("--cells", type=int, default=50000)
    ap.add_argument("--densities", default="0.05,0.10,0.30")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lcpm_sparse_bench: needs a GPU")
    from normalisr_b200 import normalisr as norm
    G, C = a.genes, a.cells
    res = {"card": card(), "genes": G, "cells": C, "iters": a.iters, "warmup": a.warmup, "e2e_reps": a.e2e_reps,
           "runs": []}
    for dens in (float(x) for x in a.densities.split(",")):
        dense = counts(G, C, dens, seed=7)
        csr = dense.to_sparse_csr()
        csr = torch.sparse_csr_tensor(csr.crow_indices(), csr.col_indices().to(torch.int32), csr.values(), (G, C))
        nnz = csr.values().numel()
        out_b = 8 * G * C
        dense_b = 2 * 4 * G * C + out_b
        csr_b = 2 * (8 * nnz + 8 * (G + 1)) + out_b
        same_dev = all(torch.equal(x, y) for x, y in zip(norm.lcpm(dense), norm.lcpm(csr)) if x is not None)
        td = time_device(lambda: norm.lcpm(dense), a.iters, a.warmup)
        ts = time_device(lambda: norm.lcpm(csr), a.iters, a.warmup)
        # the same counts as a scipy CSR matrix on the host
        h = sp.csr_matrix((csr.values().cpu().numpy(), csr.col_indices().cpu().numpy(), csr.crow_indices().cpu().numpy()),
                          shape=(G, C))
        del dense, csr
        torch.cuda.empty_cache()
        t_sp, t_de, t_toarray = [], [], []
        same_host = None
        for rep in range(a.e2e_reps + 1):                     # rep 0 warms both arms (page-locked rings, tables)
            t0 = time.perf_counter()
            r_sp = norm.lcpm(h)
            t1 = time.perf_counter()
            d = h.toarray()
            t2 = time.perf_counter()
            r_de = norm.lcpm(d)
            t3 = time.perf_counter()
            del d
            if rep == 0:
                same_host = all(np.array_equal(x, y) for x, y in zip(r_sp, r_de) if x is not None)
            else:
                t_sp.append(t1 - t0)
                t_de.append(t3 - t1)
                t_toarray.append(t2 - t1)
            del r_sp, r_de
        run = {
            "density": dens, "nnz": nnz,
            "device": {
                "dense_int32_s": float(np.median(td)), "csr_s": float(np.median(ts)),
                "dense_int32_all_s": td, "csr_all_s": ts,
                "dense_algorithmic_bytes": dense_b, "csr_algorithmic_bytes": csr_b,
                "dense_GBps": dense_b / np.median(td) / 1e9, "csr_GBps": csr_b / np.median(ts) / 1e9,
                "bit_identical": bool(same_dev)},
            "e2e_numpy_out": {
                "csr_s": float(np.median(t_sp)), "toarray_then_dense_s": float(np.median(t_de)),
                "toarray_alone_s": float(np.median(t_toarray)),
                "csr_all_s": t_sp, "toarray_then_dense_all_s": t_de,
                "host_csr_bytes": int(h.data.nbytes + h.indices.nbytes + h.indptr.nbytes),
                "host_dense_bytes": int(G * C * h.data.itemsize),
                "bit_identical": bool(same_host)},
        }
        res["runs"].append(run)
        print(json.dumps({"density": dens, "device": {k: v for k, v in run["device"].items() if "all" not in k},
                          "e2e": {k: v for k, v in run["e2e_numpy_out"].items() if "all" not in k}}), flush=True)
        del h
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ok = all(r["device"]["bit_identical"] and r["e2e_numpy_out"]["bit_identical"] for r in res["runs"])
    print(json.dumps({"card": res["card"], "all_bit_identical": ok}))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
