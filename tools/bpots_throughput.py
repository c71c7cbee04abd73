"""BP-OTS throughput, device-resident (ldpcb200_bpots_device), in syndromes/s, next to the CPU restatement.

Cases: C1 at per 0.01, 100 iterations, T 9, C 2 (the BP-OTS case of the reference's benchmark/benchmarks.jl); C4,
hgp_x(gallager(64,4,3)) and C5 at their BASELINE priors (C4's prior for the HGP code).  Each code runs on the shared-memory
path and on the global workspace (option bpots_memory = 2) wherever both apply.  Syndromes are sampled on the device
(Philox, i.i.d. errors at the prior); the timed window is CUDA events around `reps` back-to-back calls after one warm-up
call.  The CPU column is oracle.bpots_decode (C, all host threads) on a subset of the same syndromes.

    python tools/bpots_throughput.py [--quick]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

# (label, code, per, max_iters, T, C, B on the GPU, B on the CPU)
CASES = [
    ("C1", "C1", 0.01, 100, 9, 2.0, 20000, 2000),
    ("C4", "C4", 0.02, 32, 9, 2.0, 20000, 2000),
    ("hgp_x(gallager(64,4,3))", "hgp64", 0.02, 32, 9, 2.0, 4000, 400),
    ("C5", "C5", 0.02, 32, 9, 2.0, 1000, 32),
]


def matrix(pkg, code):
    if code == "hgp64":
        return pkg.codes.hgp_x(pkg.codes.gallager(64, 4, 3))
    return pkg.codes.config_matrix(code)[0]


def time_gpu(dec, B, per, seed, min_seconds):
    info = dec.info()
    SW, NW = info["syn_words"], info["err_words"]
    dev = torch.device("cuda:0")
    truth = torch.empty((B, NW), dtype=torch.int32, device=dev)
    syn = torch.empty((B, SW), dtype=torch.int32, device=dev)
    err = torch.empty((B, NW), dtype=torch.int32, device=dev)
    conv = torch.empty(B, dtype=torch.uint8, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    ctr = torch.zeros(4, dtype=torch.int64, device=dev)
    st = torch.cuda.Stream(device=dev)
    dec._bp.sample_device(B, 0, seed, per, truth.data_ptr(), syn.data_ptr(), stream=st.cuda_stream)

    def call():
        dec.decode_device(B, syn.data_ptr(), err.data_ptr(), conv.data_ptr(), iters.data_ptr(), ctr.data_ptr(), stream=st.cuda_stream)

    call()                                                     # warm-up: module load, workspace allocation
    st.synchronize()
    t0 = time.perf_counter()
    call()
    st.synchronize()
    reps = max(1, min(50, int(min_seconds / max(time.perf_counter() - t0, 1e-6))))
    ctr.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        call()
    b.record(st)
    b.synchronize()
    ms = a.elapsed_time(b)
    c = ctr.cpu().tolist()
    return dict(rate=B * reps / (ms / 1e3), ms_per_call=ms / reps, reps=reps, converged=c[1] / max(c[0], 1),
                mean_iters=c[2] / max(c[0], 1), workspace=dec.info()["bpots_workspace_bytes"], message_bytes=info["message_bytes"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small batches and short windows (a check that the script runs)")
    args = ap.parse_args()
    pkg = entry.load_package()
    oracle = entry.load_oracle()
    oracle.build()
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("device: %s (name, power limit, max SM clock); CPU restatement threads: %d" % (q.stdout.strip(), oracle.num_threads()))
    min_seconds = 0.2 if args.quick else 2.0
    for label, code, per, mi, T, C, Bg, Bc in CASES:
        if args.quick:
            Bg, Bc = min(Bg, 500), min(Bc, 8)
        H = matrix(pkg, code)
        s, n = H.shape
        need = (16 * H.nnz + 23 * n + 4 * s + 15) // 16 * 16 + 512
        cols = []
        for mem in (1, 2):
            dec = pkg.BPOTSDecoder(H, per, mi, T=T, C=C, bpots_memory=mem)
            try:
                r = time_gpu(dec, Bg, per, 97, min_seconds)
            except pkg._lib.LibraryError as e:
                if e.code != pkg._lib.EUNSUPPORTED:
                    raise
                r = None
            dec.close()
            cols.append(r)
        _, syn = oracle.sample(H, per, 97, 0, Bc)
        t0 = time.perf_counter()
        oracle.bpots_decode(H, per, mi, syn, T=T, C=C, nthreads=oracle.num_threads())
        cpu = Bc / (time.perf_counter() - t0)
        print("%s: %d x %d, E %d, per %g, max_iters %d, T %d, C %g; shared-memory need %d B" % (label, s, n, H.nnz, per, mi, T, C, need))
        for name, r in zip(("shared", "global"), cols):
            if r is None:
                print("  %-6s  does not fit" % name)
                continue
            print("  %-6s  %12.1f syndromes/s  (B %d, %.3f ms/call over %d calls, converged %.4f, mean iterations %.2f, "
                  "workspace %d B, BP message store %d B)" % (name, r["rate"], Bg, r["ms_per_call"], r["reps"], r["converged"],
                                                            r["mean_iters"], r["workspace"], r["message_bytes"]))
        if cols[0] and cols[1]:
            print("  global / shared: %.3f" % (cols[1]["rate"] / cols[0]["rate"]))
        print("  CPU restatement  %10.1f syndromes/s  (B %d)" % (cpu, Bc))
        sys.stdout.flush()


if __name__ == "__main__":
    main()
