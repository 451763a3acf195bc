#!/usr/bin/env python
"""WHICH=cholesky: times the factorisation + inverse of one 10k-wide system instead (ROWS=100000 keeps the data small).
Times ONE CSR Gram build (1M x 10k x 1 %, the bench's partition 0) through mlease_time_kernel.
Scratch tool for kernel work on a GPU box, not part of the product.  Round 2: 44.7 ms per build; 40.0 ms with producers
that only hand stages over, i.e. the MMA stream itself (power-limited clocks) is 90 % of the time."""
import os, sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "ml-ease_b200"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
import mlease_b200 as mb
import bench

n = int(os.environ.get("ROWS", 1000000)); D = 10000; nnz = 100
dev = torch.device("cuda:0")
import numpy as np
beta = (np.random.default_rng(7).normal(size=D) / np.sqrt(nnz)).astype(np.float32)
rp, ci, vv, y = bench.gen_sparse(0, n, D, nnz, beta, dev)
with mb.AdmmSession(1, D, [1.0], device=0) as s:
    s.add_partition_csr(0, rp, ci, vv, y)
    if os.environ.get("WHICH", "gram") == "cholesky":
        # factorisation + inverse of ONE 10k-wide system (TF32 merges of the inverse)
        ms = s.time_kernel(0, "cholesky", reps=3)
        print("cholesky+inverse ms per factorisation", ms)
    else:
        ms = s.time_kernel(0, "gram", reps=3)
        print("gram ms per build", ms, "PFLOP/s", n * 10016.0 * 10017.0 / ms / 1e12)
