#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark of the GenEO hot path (contract: see DESIGN.md "Measurement").

Workload (BASELINE.json configs[4], the weak-scaling unit; configs[1] does not fit one GPU, DESIGN.md "Memory"):
3-D 7-point Laplacian from the reference's own generator grammar (`--dim 3 --size S --inpEps 0.0001`,
tst/laplacian/laplacian.cpp:56-188), S^3 = 200^3 = 8.0 M DOFs and 8 subdomains PER GPU, two-level GenEO
(`-geneo_lvl ASM,1 -geneo_tau 0.1`), CG to rtol 1e-5 on the preconditioned residual.

Partition.  `--partition box` (default, every N): a 2x2x2 block of box subdomains per GPU, so that N = 1, 2, 4, 8 run
the SAME kind of partition and the weak-scaling curve compares like with like (METIS on the global 16-64 M element mesh
does not fit one rank's time or memory).  `--partition metis` (N = 1 only): the reference's METIS dual k-way partition
(src/geneo4PETSc.cpp:381-445); its parity is what tests/ pin.

One "step" = one complete pass of the hot path over the problem resident in HBM:
    numeric GenEO setup (3 sparse LDL^T factorizations + 1 block-Lanczos eigen-solve per subdomain, Z, E = Z^T A Z,
    E^-1) followed by the preconditioned Krylov solve                       -> `value` = N_dof / step seconds.
`e2e` = the same metric through the C ABI with HOST buffers: geneo_pc_create + geneo_pc_setup (host symbolic analysis,
H2D upload of every matrix, numeric setup) + geneo_ksp_solve (host b in, host x out) -- what a PETSc caller times as
"solver set up" + "solver iterations" (src/geneo4PETSc.cpp:1363-1367, 1239-1242).  Mesh generation and decomposition
(the reference does them before KSPSetUp too, src/geneo4PETSc.cpp:571-641) are reported next to it (`e2e.gen_s`,
`e2e.part_decomp_s`), not inside it.

`--impl reference` times the CPU restatement of the reference (oracle/, scipy SuperLU + ARPACK; the reference itself
needs PETSc/SLEPc/MUMPS/MPI which this image does not have) on the host cores.  Its `config.workload` names the size it
REALLY ran (the largest one that fits the time budget for the requested number of steps), and `cpu_baseline.scaling`
lists DOF/s at the smaller sizes it passed on the way, so that the size dependence is visible.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "geneo_solve_throughput(setup+iter)"
UNIT = "DOF/s"
CPU_SIZES = (24, 32, 40, 48, 56, 64, 72, 80, 96, 112, 128, 160, 200)
CPU_GRAPH_SIZES = (400, 1600, 6400, 25600, 102400, 409600, 1000000)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=0, help="grid edge per GPU (weak scaling: edge = cbrt(size^3 * gpus)), default 200; "
                                                         "--kind graph: the generator's --size (nodes per block), default 1000000")
    ap.add_argument("--kind", default="laplacian", choices=["laplacian", "heat", "graph"])
    ap.add_argument("--graph-level", type=int, default=5, help="--kind graph: levels of 4 blocks around the central block")
    ap.add_argument("--partition", default="", choices=["", "box", "metis"], help="default: box for the grids, metis for the graph")
    ap.add_argument("--subs-per-gpu", type=int, default=8)
    ap.add_argument("--lvl", default="ASM,1")
    ap.add_argument("--tau", default="0.1")
    ap.add_argument("--ksp", default="", help="cg | gmres (default: cg, gmres for --kind graph: BASELINE configs[3])")
    ap.add_argument("--rtol", type=float, default=1e-5)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-size", type=int, default=0, help="grid edge of the CPU sample; 0 = the largest that fits --cpu-budget")
    ap.add_argument("--cpu-budget", type=float, default=25.0, help="seconds of CPU work for the cpu_baseline leg of the b200 arm")
    ap.add_argument("--ref-budget", type=float, default=200.0, help="seconds for the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-opts", default="", help="more -geneo_* / -els2_* options, space separated")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step returned (solution x, its / rnorm / reason) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    graph = a.kind == "graph"
    a.size = a.size or (1000000 if graph else 200)
    a.partition = a.partition or ("metis" if graph else "box")
    a.ksp = a.ksp or ("gmres" if graph else "cg")
    if graph and a.partition != "metis":
        ap.error("--kind graph has no box partition")
    return a


def gen_args(a, size, ws=1):
    if a.kind == "graph":  # tst/graph/graphRun.sh:144
        return "--size %d --level %d --weakScaling %d --noGround --inpEps 0.0001" % (size, a.graph_level, ws)
    s = "--dim 3 --size %d --inpEps 0.0001" % size
    if a.kind == "heat":
        s += " --kappa 100. minmax --lbd 1. --dt 0.1"
    return s


def weak_edge(size, g):
    # the reference's own weak-scaling rule incl. its float truncation (tst/laplacian/laplacian.cpp:104)
    return size if g == 1 else int(math.floor((float(size) ** 3 * g) ** (1.0 / 3.0) + 1e-9))


def graph_nodes(a, size, ws=1):
    return (1 + 4 * a.graph_level) * int(math.sqrt(size * ws)) ** 2


def workload_name(a, edge, nsub, ngpu, partition):
    part = "box partition %d per GPU" % a.subs_per_gpu if partition == "box" else "METIS dual"
    if a.kind == "graph":
        return "graph Laplacian (tst/graph) size %d level %d weakScaling %d = %d nodes, %d subdomains (%s), geneo %s tau=%s, %s rtol %g" % (
            edge, a.graph_level, ngpu, graph_nodes(a, edge, ngpu), nsub, part, a.lvl, a.tau, a.ksp, a.rtol)
    return "%s3d %d^3 = %d DOFs, %d subdomains (%s), geneo %s tau=%s, %s rtol %g" % (
        a.kind, edge, edge ** 3, nsub, part, a.lvl, a.tau, a.ksp, a.rtol)


def workload_config(a, ngpu):
    graph = a.kind == "graph"
    edge = a.size if graph else weak_edge(a.size, ngpu)
    return {"workload": workload_name(a, edge, a.subs_per_gpu * ngpu, ngpu, a.partition),
            "generator": gen_args(a, edge, ngpu if graph else 1), "partition": a.partition,
            "l2": "inputs_larger_than_L2 (factors >> 126 MB)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md, "clocks line")."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            self.th.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle = test infrastructure; used here ONLY as the timed CPU baseline / checker, never on the product path)
# ---------------------------------------------------------------------------------------------------------------------
def box_elem_part(mesh, edge, K):
    """Box partition of the generator's elements in numpy (element -> box of its first = lower node), the rule of
    geneo_problem_generate_boxed restated for the oracle."""
    import numpy as np
    first = np.asarray(mesh.elem_idx)[np.asarray(mesh.elem_ptr[:-1])]
    d1, d2, d3 = first % edge, (first // edge) % edge, first // (edge * edge)
    b = (d1 * K[0]) // edge + K[0] * ((d2 * K[1]) // edge + K[1] * ((d3 * K[2]) // edge))
    return b.astype(np.int32)


def cpu_sample(a, size, nparts, partition):
    """One setup+solve of the CPU restatement on `size`^3 DOFs; returns (report, dofs, seconds, cores, partition arrays)."""
    import numpy as np
    from oracle import geneo_oracle as go
    from geneo4petsc_b200.dist import box_dims
    if a.kind == "graph":  # (the reference's own generator, compiled into oracle/_ref)
        mesh = go.ref_generator("graph", gen_args(a, size))
    else:
        kappa, interp = (100.0, "minmax") if a.kind == "heat" else (1.0, "")
        mesh = go.gen_grid(3, size, 1e-4, kappa, interp, heat=(a.kind == "heat"))
    l1, l2 = a.lvl.split(",")
    cores = max(1, min(nparts, os.cpu_count() or 1))  # one worker per subdomain = the reference's one MPI rank per subdomain
    if partition == "box":
        part = (box_elem_part(mesh, size, box_dims(nparts)), np.zeros(mesh.nb_node, dtype=np.int32))
    else:
        part = go.metis_partition(mesh, nparts, True)
    rep = go.run_case(mesh, nparts, go.GenEOOptions(lvl1=l1, lvl2=l2, tau=float(a.tau)), ksp=a.ksp, rtol=a.rtol, workers=cores, part=part)
    rep.part = part
    return rep, mesh, rep.setup_s + rep.solve_s, cores


def cpu_ladder(a, nparts, partition, budget, repeats=1, fixed=0):
    """Walk up CPU_SIZES while (predicted time of the next size) x repeats fits the budget.  Returns
    (table [(size, dofs, seconds, its)], last report, last mesh, cores).  The time of the next size is extrapolated with the
    measured exponent of the last two (sparse direct solvers are super-linear in the DOFs)."""
    table, rep, mesh, cores = [], None, None, 1
    spent = 0.0
    sizes = [fixed] if fixed else list(CPU_GRAPH_SIZES if a.kind == "graph" else CPU_SIZES)
    for i, s in enumerate(sizes):
        rep, mesh, secs, cores = cpu_sample(a, s, nparts, partition)
        table.append((s, mesh.nb_node, secs, rep.ksp.its))
        spent += secs
        if i + 1 >= len(sizes):
            break
        expo = 1.6
        if len(table) >= 2 and table[-2][2] > 0.2:
            expo = max(1.2, min(2.2, math.log(table[-1][2] / table[-2][2]) / math.log(table[-1][1] / table[-2][1])))
        grow = (sizes[i + 1] / float(s)) if a.kind == "graph" else (sizes[i + 1] ** 3 / float(s ** 3))
        pred = secs * grow ** expo
        if spent + pred * repeats > budget:
            break
    return table, rep, mesh, cores


def scaling_rows(table):
    return [{"edge": s, "dofs": n, "seconds": round(t, 3), "its": its, "dofs_per_s": round(n / t, 1)} for (s, n, t, its) in table]


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nparts = a.subs_per_gpu
    reps = max(1, a.steps + a.warmup)
    # ladder: one pass per size up to the largest edge whose (steps + warmup) repetitions fit the budget ...
    table, rep, mesh, cores = cpu_ladder(a, nparts, a.partition, a.ref_budget, repeats=reps, fixed=a.cpu_size)
    size = table[-1][0]
    # ... then the timed steps at that size (the ladder pass was the first warm-up)
    vals, its = [], table[-1][3]
    for i in range(max(0, a.warmup - 1) + a.steps):
        rep, mesh, secs, cores = cpu_sample(a, size, nparts, a.partition)
        if i >= max(0, a.warmup - 1):
            vals.append(secs)
        its = rep.ksp.its
    t = sum(vals) / len(vals)
    n = mesh.nb_node
    v = n / t
    wl = workload_name(a, size, nparts, 1, a.partition)
    sample = "%s: scipy SuperLU/ARPACK restatement of the reference (PETSc/MUMPS/SLEPc absent), %d worker threads, %d its, dimE %d" % (
        wl, cores, its, rep.pc.e.shape[0] if rep.pc.e is not None else 0)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": wl, "generator": gen_args(a, size), "partition": a.partition,
                   "note": "CPU sample: the edge is the largest whose steps+warmup repetitions fit %.0f s; the b200 arm runs %d^3 per GPU -- "
                           "a ratio of the two values is a CROSS-SIZE ratio (see cpu_baseline.scaling and the b200 arm's parity.same_size)"
                           % (a.ref_budget, a.size)},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "scaling": scaling_rows(table)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---------------------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------------------
def dgemm_peak(torch, n=6144, reps=4):
    """FP64 GEMM throughput of the library GEMM (cuBLAS through torch.matmul) measured in this run: the practical
    denominator of the factorization roofline (MEASURED_PEAKS.json holds no FP64 number)."""
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    torch.cuda.empty_cache()
    return best


def build_problem(a, g, dist, rank, world, edge, partition):
    """Generate + partition + decompose; returns (problem, layout | None, timings)."""
    t0 = time.time()
    prob = g.Problem()
    layout = None
    if partition == "box":
        K, rg, sub_rank = dist.box_grid(world, a.subs_per_gpu)
        lo, hi = dist.keep_region(edge, K, rg, rank, a.subs_per_gpu) if world > 1 else (None, None)
        e2 = dist.generate_boxed(prob, a.kind, gen_args(a, edge), K, lo, hi)
        assert e2 == edge, (e2, edge)
        t1 = time.time()
        dist.decompose_owned(prob, len(sub_rank), sub_rank, rank, True, 0)
        if world > 1:
            layout = dist.Layout(prob, rank, world, sub_rank)
    else:  # the reference's METIS dual partition; N > 1: every rank partitions the same mesh, parts grouped onto the GPUs
        prob.generate(a.kind, gen_args(a, edge, world if a.kind == "graph" else 1))
        t1 = time.time()
        if world == 1:
            prob.decompose(a.subs_per_gpu, True, 0)
        else:
            sub_rank = dist.metis_problem(prob, a.subs_per_gpu * world, world, rank)
            layout = dist.Layout(prob, rank, world, sub_rank)
    t2 = time.time()
    return prob, layout, {"gen_s": t1 - t0, "part_decomp_s": t2 - t1}


DUMP_X_MAX = 1 << 21  # rows of x written by --dump-outputs: 2 x 16 MB with their ids


def dump_outputs(d, x, r):
    """The result of the last timed step as float64 .npy files: x (the solution; above DUMP_X_MAX rows a fixed seeded sample
    of them, whose row ids are x_index) and ksp = [iterations, rnorm, reason]."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    n = x.shape[0]
    idx = np.arange(n) if n <= DUMP_X_MAX else np.sort(np.random.default_rng(0).choice(n, DUMP_X_MAX, replace=False))
    np.save(os.path.join(d, "x.npy"), x[idx])
    np.save(os.path.join(d, "x_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, "ksp.npy"), np.array([r["its"], r["rnorm"], r["reason"]], dtype=np.float64))


def run_b200(a):
    import numpy as np
    import torch
    import geneo4petsc_b200 as g
    from geneo4petsc_b200 import dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    if a.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes the solution of a single process; run it on one GPU")
    torch.cuda.set_device(local)
    tdist = None
    if world > 1:
        import torch.distributed as tdist
        tdist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))

    def barrier():
        if tdist is not None:
            tdist.barrier()

    edge = a.size if a.kind == "graph" else weak_edge(a.size, world)
    prob, layout, tprob = build_problem(a, g, dist, rank, world, edge, a.partition)
    n = prob.sizes()["nb_node"]
    extra = a.extra_opts.split() if a.extra_opts else []
    opts = ["-geneo_lvl", a.lvl, "-geneo_tau", a.tau, "-geneo_kernel_timing"] + extra

    def new_pc(options):
        pc = g.GeneoPC(options)
        if layout is not None:
            layout.exchange_requests(tdist)
            dist.setup_dist(pc, prob, layout, dist.nccl_unique_id(tdist, rank))
        else:
            pc.setup(prob)
        return pc

    pc = new_pc(opts)  # cold: host symbolic + upload + numeric
    tm_cold = pc.timers()
    st = pc.stats()
    n_own, n_loc = dist.local_sizes(pc)
    x = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    b = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    ones = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
    if layout is not None:
        ones[:n_own] = torch.from_numpy(layout.owned.astype(np.float64) + 1.0).cuda()
    else:
        ones = torch.arange(1, n + 1, dtype=torch.float64, device="cuda")
    pc.mult_device(ones.data_ptr(), b.data_ptr())  # b = A (1..N), src/geneo4PETSc.cpp:820-831
    torch.cuda.synchronize()

    def step():
        pc.refactor()
        return pc.ksp_solve_device(b.data_ptr(), x.data_ptr(), ksp=a.ksp, rtol=a.rtol, atol=1e-50, restart=30)

    for _ in range(a.warmup):
        r = step()
    torch.cuda.synchronize()
    pc.kernel_time()
    c0 = g.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    setup_s = iter_s = fac_s = fac_f = 0.0
    with ClockSampler(local) as clk:
        barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.steps):
            ta = time.perf_counter()
            pc.refactor()
            tb = time.perf_counter()
            r = pc.ksp_solve_device(b.data_ptr(), x.data_ptr(), ksp=a.ksp, rtol=a.rtol, atol=1e-50, restart=30)
            tc = time.perf_counter()
            setup_s += tb - ta
            iter_s += tc - tb
            fs = pc.factor_stats()
            fac_s += fs["seconds"]
            fac_f += fs["flops"]
        e1.record()
        torch.cuda.synchronize()
        barrier()
    ms = e0.elapsed_time(e1) / a.steps
    c1 = g.counters()
    kms, klaunch = pc.kernel_time()
    assert r["reason"] > 0, "KSP did not converge: %s" % r["reason_name"]
    err = float((x[:n_own] - ones[:n_own]).abs().max() / n)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, x[:n_own].cpu().numpy(), r)
    phases = {k: pc.timers()[k] for k in ("lvl1SetupMinv", "lvl2SetupSyl", "lvl2SetupEig", "lvl2SetupZ", "lvl2SetupE")}
    info = pc.info()

    # PC-apply and SpMV alone (device pointers), algorithmic GB/s of this rank
    rates = {}
    y = torch.empty_like(x)
    for name, fn, nbytes in (("pc_apply", pc.apply_device, st["apply_bytes"]), ("spmv", pc.mult_device, st["spmv_bytes"])):
        for _ in range(3):
            fn(b.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(10):
            fn(b.data_ptr(), y.data_ptr())
        f1.record()
        torch.cuda.synchronize()
        t = f0.elapsed_time(f1) / 10
        rates[name] = {"ms": t, "GBps": nbytes / t / 1e6}
    pc.kernel_time()
    # the factorization kernels alone: every level-1 matrix factorized once more (same values), CUDA events around the lot
    pc.factor_bench()
    fb_s, fb_f = pc.factor_bench()
    del pc, y, fn, step  # the e2e leg below builds a second preconditioner from scratch: this one's factors and workspaces must
    #                      go first (fn / step hold bound references to it)
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    gemm_tf = dgemm_peak(torch) if rank == 0 else 0.0

    # end to end through the C ABI with host buffers: create + setup (host analysis, uploads, numeric) + solve
    bh = b.cpu().numpy()
    e2e_t, h2d, d2h = [], 0, 0
    tm2, fs2 = {"symbolic": 0.0, "upload": 0.0, "numeric": 0.0}, {"ordering_reuse_s": 0.0}
    for _ in range(max(1, a.e2e_steps)):
        barrier()
        torch.cuda.synchronize()
        k0 = g.counters()
        ta = time.perf_counter()
        pc2 = new_pc(["-geneo_lvl", a.lvl, "-geneo_tau", a.tau] + extra)
        r2 = pc2.ksp_solve(bh, ksp=a.ksp, rtol=a.rtol, atol=1e-50, restart=30)
        torch.cuda.synchronize()
        tb = time.perf_counter()
        k1 = g.counters()
        e2e_t.append(tb - ta)
        h2d, d2h = k1["h2d"] - k0["h2d"], k1["d2h"] - k0["d2h"]
        tm2, fs2 = pc2.timers(), pc2.factor_stats()
        assert r2["reason"] > 0
        del pc2
    e2e_s = sum(e2e_t) / len(e2e_t)

    kavg = kms / max(1, klaunch)
    launches = float(c1["launches"] - c0["launches"])
    tri_b, fac_b, fac_fl = st["trisolve_bytes"], st["factor_bytes"], st["factor_flops"]
    if tdist is not None:  # max over ranks of the times, sums of the per-rank statistics
        red = torch.tensor([ms, e2e_s, err, kavg, fac_s, tm2["symbolic"], tm2["numeric"], tprob["part_decomp_s"], tprob["gen_s"]],
                           dtype=torch.float64, device="cuda")
        tdist.all_reduce(red, op=tdist.ReduceOp.MAX)
        ms, e2e_s, err, kavg_max, fac_s_max, sym_max, num_max, pd_max, gen_max = [float(v) for v in red.cpu()]
        sums = torch.tensor([tri_b, fac_b, fac_fl, float(h2d), float(d2h), launches, fac_f], dtype=torch.float64, device="cuda")
        tdist.all_reduce(sums, op=tdist.ReduceOp.SUM)
        tri_b_tot, fac_b, fac_fl, h2d, d2h, launches, fac_f_tot = [float(v) for v in sums.cpu()]
    else:
        kavg_max, fac_s_max, sym_max, num_max, pd_max, gen_max = kavg, fac_s, tm2["symbolic"], tm2["numeric"], tprob["part_decomp_s"], tprob["gen_s"]
        tri_b_tot, fac_f_tot = tri_b, fac_f
    if rank != 0:
        barrier()
        tdist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    ach = tri_b / kavg / 1e6 if kavg > 0 else 0.0  # rank 0's kernel against one GPU's HBM
    cfg = workload_config(a, world)
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of THIS workload
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(cfg["workload"])
    except (OSError, ValueError):
        pass
    fac_tf = fb_f / fb_s / 1e12 if fb_s > 0 else 0.0  # rank 0, factorization kernels timed alone
    pipe_tf = fac_f / fac_s / 1e12 if fac_s > 0 else 0.0  # rank 0, inside the step (eigen-solves share the device)
    out = {
        "metric": METRIC, "value": n / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "clocks": clk.summary(),
        "e2e": {"value": n / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "seconds": e2e_s,
                "seconds_runs": [round(t, 3) for t in e2e_t],
                "symbolic_s": sym_max, "upload_s": tm2["upload"], "numeric_s": num_max, "ordering_reuse_s": fs2["ordering_reuse_s"],
                "gen_s": gen_max, "part_decomp_s": pd_max,
                "note": "seconds = create + setup (host analysis, H2D, numeric) + solve with host b/x; gen_s / part_decomp_s (mesh "
                        "generation, partition + decomposition: before KSPSetUp in the reference too) are reported, not included"},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "k_solve_ring<1> (level-1 triangular sweeps of all local subdomains, one launch per PC apply; rank 0)",
                     "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (copy)" if peaks else "fallback 6650",
                     "traffic": traffic, "algorithmic_bytes_per_launch": tri_b, "launches_timed": klaunch, "avg_launch_ms": kavg},
        "roofline_factorization": {
            "kernel": "block LDL^T factorization kernels (k_schur2 / k_schur / k_panel DMMA tiles, k_diag_invert, assembly): the level-1 "
                      "factorizations of all local subdomains, alone on the device, rank 0",
            "bound": "tensor", "achieved": fac_tf, "peak": gemm_tf, "unit": "TFLOP/s", "frac": fac_tf / gemm_tf if gemm_tf else None,
            "peak_source": "cuBLAS DGEMM 6144^3 through torch.matmul measured in this run (no FP64 entry in MEASURED_PEAKS.json; "
                           "nominal FP64 tensor peak of B200 ~ 37-40 TFLOP/s)",
            "flops_timed": fb_f, "seconds_timed": fb_s,
            "in_step": {"flops_per_step": fac_f / a.steps, "pipeline_span_s_per_step": fac_s / a.steps, "TFLOPs": pipe_tf,
                        "share_of_step": fac_s / a.steps / (ms * 1e-3),
                        "note": "span of the factorization pipeline inside the timed steps: 3 factorizations per subdomain on several "
                                "streams; the block-Lanczos eigen-solves run inside the same span and take the SMs in turn"},
            "how": "flops = sum over fronts of k^3/3 + m k^2 + m^2 k (symbolic analysis); achieved = the level-1 factorizations of all "
                   "local subdomains run once more, alone on the device, between two CUDA events (geneo_pc_factor_bench)"},
        "detail": {"n_dof": n, "iterations": r["its"], "reason": r["reason_name"], "rnorm": r["rnorm"], "max_rel_err_vs_1..N": err,
                   "setup_numeric_s": setup_s / a.steps, "iter_s": iter_s / a.steps, "dimE": info["nE"],
                   "nev_min_max": [info["realMin"], info["realMax"]],
                   "cold_setup_rank0": {k: tm_cold[k] for k in ("symbolic", "upload", "numeric", "operator", "setup")},
                   "numeric_phases_s_rank0": phases, "rank0_local": {"n_own": n_own, "n_ghost": n_loc - n_own},
                   "factor_bytes_total": fac_b, "factor_flops_total": fac_fl, "trisolve_bytes_total": tri_b_tot,
                   "pc_apply_rank0": rates["pc_apply"], "spmv_rank0": rates["spmv"], "hbm_peak_GBps": peak, "dgemm_TFLOPs": gemm_tf},
    }
    if not a.no_cpu_baseline and world == 1:
        # CPU restatement on a bounded sample of the same workload + the GPU on that SAME sample: a same-size ratio and a
        # parity point (iterations, coarse dimension, eigen-counts) for free
        table, rep, mesh, cores = cpu_ladder(a, a.subs_per_gpu, a.partition, a.cpu_budget, fixed=a.cpu_size)
        s_edge, nn, secs, its = table[-1]
        out["cpu_baseline"] = {"value": nn / secs, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "%s (%d its, %.1f s): scipy SuperLU/ARPACK restatement of the reference (PETSc/MUMPS/SLEPc "
                                         "absent), %d worker threads" % (workload_name(a, s_edge, a.subs_per_gpu, 1, a.partition), its, secs, cores),
                               "scaling": scaling_rows(table)}
        p3 = g.Problem().set_mesh(mesh.nb_node, mesh.elem_ptr, mesh.elem_idx, mesh.mat_val)
        p3.decompose(a.subs_per_gpu, True, 0, elem_part=rep.part[0])
        gpu_t = []
        for _ in range(2):  # twice: the first run of a fresh handle pays for pinned buffers, streams and the lanes' allocations
            torch.cuda.synchronize()
            ta = time.perf_counter()
            pc3 = g.GeneoPC(["-geneo_lvl", a.lvl, "-geneo_tau", a.tau] + extra).setup(p3)
            b3 = rep.b
            r3 = pc3.ksp_solve(b3, ksp=a.ksp, rtol=a.rtol, atol=1e-50, restart=30)
            tb = time.perf_counter()
            gpu_t.append(tb - ta)
        est_gpu = [pc3.sub_info(s)["estim"] for s in range(a.subs_per_gpu)]
        est_cpu = [int(s.estim) for s in rep.pc.sub]
        out["parity"] = {"sample": "size %d, same partition arrays, same options" % s_edge,
                         "its_gpu": r3["its"], "its_cpu": its, "dimE_gpu": pc3.info()["nE"], "dimE_cpu": int(rep.pc.e.shape[0]),
                         "eigen_counts_equal": est_gpu == est_cpu,
                         "x_rel_diff": float(np.linalg.norm(r3["x"] - rep.ksp.x) / np.linalg.norm(rep.ksp.x)),
                         "same_size": {"edge": s_edge, "gpu_e2e_dofs_per_s": nn / gpu_t[0], "gpu_e2e_dofs_per_s_second_run": nn / gpu_t[1],
                                       "cpu_dofs_per_s": nn / secs, "ratio": secs / gpu_t[0], "ratio_second_run": secs / gpu_t[1]}}
        del pc3
    print(json.dumps(out), flush=True)
    if os.environ.get("GENEO_PROFILE"):
        g.profile_dump(os.environ.get("GENEO_PROFILE_OUT", "gpurun_out/profile_sites.csv"))
    if tdist is not None:
        barrier()
        tdist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
