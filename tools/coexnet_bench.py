#!/usr/bin/env python3
"""The co-expression network from a numpy expression matrix (default 100,000 cells x 20,000 genes, the
planted-module recipe of bench.py with its seed, qcut 0.05), three ways, on one GPU and on all GPUs of the box:

  coex+binnet   norm.coex(dt, dc) (P and dot to the host), then norm.binnet(P, qcut) (P back to one GPU)
  coexnet       norm.coexnet(dt, dc, qcut): the dense bool network, P and dot stay on the GPUs
  coexnet_csr   norm.coexnet(dt, dc, qcut, sparse=True): the network as a scipy CSR matrix

Host clock around whole calls (each ends with its results on the host), the arms alternated, after one warm-up
call of each.  The networks of all arms are compared bit for bit in the same run.  Bytes moved each way across
PCIe are counted from the shapes (inputs in; P, dot, var and the network out).  On one GPU it also times
norm.binnet(P, qcut, sparse=True) against the dense norm.binnet on a device-resident P (CUDA events).
The card's name and power limit are recorded beside the numbers.
python tools/coexnet_bench.py --out profiles/coexnet_b200.json"""
import argparse
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


def net_bytes(net):
    if isinstance(net, np.ndarray):
        return net.nbytes
    return net.indptr.nbytes + net.indices.nbytes


def same_net(a, b):
    if isinstance(a, np.ndarray) != isinstance(b, np.ndarray):
        if isinstance(a, np.ndarray):
            a, b = b, a
        import scipy.sparse
        b = scipy.sparse.csr_matrix(b)
    if isinstance(a, np.ndarray):
        return bool(np.array_equal(a, b))
    return bool(np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices))


def device_binnet(P, qcut, reps):
    """binnet(sparse=True) against dense binnet on a device-resident P: ms per call (CUDA events, results on
    the device)."""
    from normalisr_b200 import normalisr as norm
    out = {}
    for name, sparse in (("dense", False), ("csr", True)):
        for _ in range(2):
            norm.binnet(P, qcut, sparse=sparse)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            net = norm.binnet(P, qcut, sparse=sparse)
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        out[name + "_ms"] = ts
        out[name + "_bytes"] = net.numel() if not sparse else sum(t.numel() * t.element_size()
                                                                  for t in (net.crow_indices(), net.col_indices()))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--genes", type=int, default=20000)
    ap.add_argument("--cells", type=int, default=100000)
    ap.add_argument("--qcut", type=float, default=0.05)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("coexnet_bench: needs a GPU")
    from normalisr_b200 import normalisr as norm, synth
    G, C, q = a.genes, a.cells, a.qcut
    p = synth.device_problem(SEED, G, C, "cuda:0")
    dt, dc = p["dt"].cpu().numpy(), p["dc"].cpu().numpy()
    del p
    torch.cuda.empty_cache()
    res = {"card": card(), "genes": G, "cells": C, "qcut": q, "reps": a.reps,
           "input_bytes_h2d": dt.nbytes + dc.nbytes, "configs": {}}

    configs = [("1gpu", None)] + ([("all", "all")] if torch.cuda.device_count() > 1 else [])
    for cname, devices in configs:
        def coex_binnet():
            P, D, var = norm.coex(dt, dc, devices=devices)
            return norm.binnet(P, q)

        arms = {"coex+binnet": coex_binnet,
                "coexnet": lambda: norm.coexnet(dt, dc, q, devices=devices)[0],
                "coexnet_csr": lambda: norm.coexnet(dt, dc, q, sparse=True, devices=devices)[0]}
        nets, times = {}, {k: [] for k in arms}
        for k, fn in arms.items():                 # warm-up, and the results compared below
            nets[k] = fn()
        for _ in range(a.reps):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                times[k].append(time.perf_counter() - t0)
        ref = nets["coex+binnet"]
        nnz = int(ref.sum())
        pg = 8 * G * G
        out = {"times_s": times, "median_s": {k: float(np.median(v)) for k, v in times.items()},
               "nnz": nnz, "identical": {k: same_net(ref, v) for k, v in nets.items()},
               "d2h_bytes": {"coex+binnet": 2 * pg + 8 * G + G * G, "coexnet": G * G + 8 * G,
                             "coexnet_csr": net_bytes(nets["coexnet_csr"]) + 8 * G},
               "h2d_bytes": {"coex+binnet": dt.nbytes + dc.nbytes + pg, "coexnet": dt.nbytes + dc.nbytes,
                             "coexnet_csr": dt.nbytes + dc.nbytes}}
        res["configs"][cname] = out
        print(cname, json.dumps({k: out[k] for k in ("median_s", "nnz", "identical")}), flush=True)
        del nets, ref

    # binnet on a device-resident P (the P of this problem on GPU 0)
    P_dev = torch.from_numpy(norm.coex(dt, dc)[0]).cuda()
    res["device_binnet"] = device_binnet(P_dev, q, 5)
    print("device_binnet", json.dumps({k: v for k, v in res["device_binnet"].items()}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
