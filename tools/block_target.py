"""Blocks of right-hand sides on the bench's workload: 200^3 Laplacian (--kappa 2 lin), 8 box subdomains, geneo ASM,1 tau 0.1,
one GPU.  Measures, in one process:
  - apply_block_device for k = 1, 8, 16, 64 columns against k single apply_device calls (CUDA events, warm-up first);
  - the 8-column solve kernel (k_solve_ring<8>) alone: its time per 8-column pass from a torch.profiler trace of a few
    block applies, and trisolve_algo_bytes (the factor stream of one pass) over that time;
  - an 8-column block CG (rtol 1e-5) against 8 sequential ksp_solve_device: wall time and per-column iterations.
Every working set is far above the 126 MB of L2 (the level-1 factors alone are tens of GB).  The card's name and power limit
are read in the same run.  Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import re
import subprocess
import sys
import time


sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import geneo4petsc_b200 as g  # noqa: E402
from geneo4petsc_b200 import dist  # noqa: E402

OPTS = ["-geneo_lvl", "ASM,1", "-geneo_tau", "0.1"]


def gpu_name_and_power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, limit = [s.strip() for s in out[0].split(",")]
        return name, limit
    except Exception as e:  # (the numbers are still printed; without the card they are not worth much)
        return "unknown (%s)" % e, "unknown"


def event_ms(torch, fn, reps):
    """mean ms of fn() over reps calls, CUDA events around the whole loop (fn enqueues on the library's stream)"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=200)
    ap.add_argument("--out", default=None, help="JSON output (default profiles/block_target_<size>.json)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available() or g.device_count() < 1:
        raise SystemExit("block_target: no CUDA device -- nothing to measure")
    gpu, power = gpu_name_and_power_limit()
    prob = g.Problem()
    K, _, sub_rank = dist.box_grid(1, 8)
    edge = dist.generate_boxed(prob, "laplacian", "--dim 3 --size %d --inpEps 0.0001 --kappa 2 lin" % a.size, K)
    dist.decompose_owned(prob, len(sub_rank), sub_rank, 0, True, 0)
    t = time.perf_counter()
    pc = g.GeneoPC(OPTS).setup(prob)
    t_setup = time.perf_counter() - t
    n = pc.info()["nbDof"]
    st = pc.stats()
    res = dict(workload="%d^3 laplacian, 8 box subdomains, %s" % (edge, " ".join(OPTS)), gpu=gpu, power_limit=power, n=n,
               dimE=pc.info()["nE"], setup_s=round(t_setup, 2), trisolve_algo_bytes=st["trisolve_bytes"])

    kmax = 64
    X = torch.randn((kmax, n), dtype=torch.float64, device="cuda")  # column-major (n, kmax), ld n
    Y = torch.zeros_like(X)
    y = torch.zeros(n, dtype=torch.float64, device="cuda")
    # single applies: warm-up, then the mean over 10 calls
    pc.apply_device(X[0].data_ptr(), y.data_ptr())
    t_single = event_ms(torch, lambda: pc.apply_device(X[0].data_ptr(), y.data_ptr()), 10)
    res["apply_ms"] = round(t_single, 3)
    cols = {}
    for k in (1, 8, 16, 64):
        pc.apply_block_device(X.data_ptr(), Y.data_ptr(), k, n, n)  # warm-up (the first 8-column call builds its item lists)
        reps = max(3, 32 // k)
        tb = event_ms(torch, lambda: pc.apply_block_device(X.data_ptr(), Y.data_ptr(), k, n, n), reps)
        seq = None
        if k == 8:  # k single applies in sequence, measured as such
            def eight():
                for j in range(8):
                    pc.apply_device(X[j].data_ptr(), y.data_ptr())
            seq = event_ms(torch, eight, 3)
        cols[str(k)] = dict(block_ms=round(tb, 3), singles_ms=round(seq if seq is not None else k * t_single, 3),
                            singles_measured=seq is not None, speedup=round((seq if seq is not None else k * t_single) / tb, 3))
    res["apply_block"] = cols

    # the 8-column solve kernel alone, from a trace of 4 block applies of 8 columns (run after the timed windows)
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(4):
            pc.apply_block_device(X.data_ptr(), Y.data_ptr(), 8, n, n)
        torch.cuda.synchronize()
    ring = [e for e in prof.events() if re.search(r"k_solve_ring<8", e.name) and str(e.device_type).endswith("CUDA")]
    if ring:
        us = sum(e.time_range.elapsed_us() for e in ring) / len(ring)
        res["solve8_kernel_ms"] = round(us / 1e3, 3)
        res["solve8_kernel_launches"] = len(ring)
        res["solve8_factor_stream_TBps"] = round(st["trisolve_bytes"] / (us * 1e-6) / 1e12, 3)
    else:
        res["solve8_kernel_ms"] = None  # (the trace held no kernel of that name)

    # block CG on 8 columns against 8 sequential CG solves
    ncg = 8
    B = torch.zeros((ncg, n), dtype=torch.float64, device="cuda")
    v = torch.zeros(n, dtype=torch.float64, device="cuda")
    ids = torch.arange(1, n + 1, dtype=torch.float64, device="cuda")
    for j in range(ncg):
        v.copy_(ids if j == 0 else torch.sin(ids * (0.37 * j)))
        pc.mult_device(v.data_ptr(), B[j].data_ptr())  # b_0 = A (1..N) as bench.py, then A sin(0.37 j i)
    Xb = torch.zeros_like(B)
    torch.cuda.synchronize()
    t = time.perf_counter()
    rb = pc.ksp_solve_block_device(B.data_ptr(), Xb.data_ptr(), ncg, n, n, ksp="cg", rtol=1e-5, atol=1e-50)
    torch.cuda.synchronize()
    t_block = time.perf_counter() - t
    its_seq, t_seq, diff = [], 0., 0.
    xs = torch.zeros(n, dtype=torch.float64, device="cuda")
    for j in range(ncg):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = pc.ksp_solve_device(B[j].data_ptr(), xs.data_ptr(), ksp="cg", rtol=1e-5, atol=1e-50)
        torch.cuda.synchronize()
        t_seq += time.perf_counter() - t
        its_seq.append(r["its"])
        diff = max(diff, float(torch.linalg.norm(Xb[j] - xs) / torch.linalg.norm(xs)))
    res["block_cg"] = dict(k=ncg, block_s=round(t_block, 3), sequential_s=round(t_seq, 3), speedup=round(t_seq / t_block, 3),
                           its_block=[int(i) for i in rb["its"]], its_sequential=its_seq,
                           reasons=[int(r) for r in rb["reason"]], max_rel_x_diff=diff)
    line = json.dumps(res)
    print(line)
    out = a.out or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                "block_target_%d.json" % a.size)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
