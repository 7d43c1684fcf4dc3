#!/usr/bin/env python
"""bench.py -- curl-curl + mass operator apply throughput (BASELINE.json metric: MDoF/s).

One "step" = one y = A x of the matrix-free ND curl-curl+mass operator on the L-vector of one
mesh partition (ceed::Operator::Mult semantics: zero-fill + apply-add), synthetic uniform hex
mesh, p = 3, ~2M dofs per GPU (BASELINE configs[1]). `value` times the device path with inputs
resident in HBM; `e2e` times the same call through the C ABI with HOST buffers (pinned host x ->
device, apply, device y -> host) every step. `--impl reference` times the reference's own
algorithm (dense non-tensor basis, the CPU oracle port) on the host cores.

Launch:  python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR]   or, for N > 1,
         python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the y of the last timed step as DIR/y.npy (DIR/y_rank<r>.npy per rank for N > 1), float64. x, the mesh
and the coefficients are fixed by the arguments, so two builds can be compared output for output, and the two arms with each other.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree may be read-only: no bytecode caches from this process or the experiments' child processes
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

METRIC = "curl-curl+mass operator apply throughput"
UNIT = "MDoF/s"
DUMP_BYTES = 64 << 20  # --dump-outputs: at most this much over all ranks


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b2p", choices=["b2p", "reference"])
    ap.add_argument("--order", type=int, default=3)
    ap.add_argument("--n", type=int, default=29, help="elements per direction per GPU (29 -> 2.02M dofs at p=3)")
    ap.add_argument("--assemble-qdata", type=int, default=0)
    ap.add_argument("--warp", type=float, default=0.0)
    ap.add_argument("--coefficient", default="iso", choices=["iso", "matrix4"],
                    help="iso: one material, identity tensors (SURVEY 8d.2 case 1); matrix4: four striped materials with full 3x3 "
                         "tensors, as the reference's unit test builds them (test/unit/test-libceed.cpp:144-168)")
    ap.add_argument("--cpu-sample-elems", type=int, default=0, help="elements in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-experiments", action="store_true", help="skip the opt-in kernel variants measured in subprocesses")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output vector of the last timed step to DIR/y.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(path, y, rank, world):
    """y (the vector the timed Mult returned) as path/y.npy, or path/y_rank<r>.npy for world > 1, float64. When y is larger than
    the rank's share of DUMP_BYTES, a fixed sample of its entries is written instead (sorted indices drawn from default_rng(0));
    the default workload's y (2.0M dofs, 16 MB) is written whole."""
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    keep = DUMP_BYTES // world // y.itemsize
    if y.size > keep:
        y = y[np.sort(np.random.default_rng(0).choice(y.size, keep, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "y.npy" if world == 1 else f"y_rank{rank}.npy"), y)


def build_problem(n, p, warp, mesh_order=1, origin=(0.0, 0.0, 0.0), size=(1.0, 1.0, 1.0), coefficient="iso"):
    from palace_b200.host import coeff as cf
    from palace_b200.host import hexmesh as hm
    from palace_b200.host import hexspace as hs

    n_attr = 4 if coefficient == "matrix4" else 1
    mesh = hm.box_mesh(n, size, warp_amp=warp, n_attr=n_attr, origin=origin)
    topo = hs.build_topology(mesh)
    nd = hs.build_nd_space(mesh, topo, p)
    q1d = p + 1
    nodes = hs.gauss_lobatto(mesh_order + 1)
    xe = mesh.node_coords(mesh_order, nodes)
    qx, qw = hs.gauss_legendre(q1d)
    nB, nG = hs.lagrange_table(nodes, qx)
    tabs = hs.tables_1d(p, q1d)
    if coefficient == "matrix4":
        # four striped materials, symmetric positive definite 3x3 tensors (the reference's unit-test coefficient,
        # test/unit/test-libceed.cpp:144-168); the curl part takes the materials in reverse order, transposed
        am, mc = cf.test_suite_coefficient(n_attr, "matrix")
        blob = cf.coeff_ctx_pair(cf.coeff_ctx(am, mc, a=1.0), cf.coeff_ctx(am, mc[::-1].copy(), a=1.0, transpose=True))
    else:
        # one material: mu^-1 = I (curl part), eps = 1 (mass part)  (SURVEY §8d.2)
        blob = cf.coeff_ctx_pair(cf.coeff_ctx(a=1.0), cf.coeff_ctx(a=1.0))
    return dict(mesh=mesh, topo=topo, nd=nd, q1d=q1d, xe=xe, nB=nB, nG=nG, tabs=tabs, blob=blob, mesh_order=mesh_order, p=p)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_quota():
    """CPUs' worth of time the container may use per scheduling period (cgroup CFS quota), or None when unlimited. Running
    more busy threads than this makes the kernel throttle the whole process for the rest of every period (measured on the
    bench box: 64 pinned threads gave 19.6 ms best / 91 ms median per step), so the reference arm sizes its pool to it."""
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()[:2]
            return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
            q = float(f.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
            per = float(f.read())
        return None if q <= 0 else q / per
    except Exception:
        return None


class CpuReference:
    """The reference algorithm (dense [3Q x P] interp/curl per element + reference QFunction arithmetic: the oracle port of
    the libCEED /cpu/self path) on the host cores, organised like libCEED's blocked CPU backend: blocks of 8 elements with
    the element index innermost, a persistent pool of threads pinned one per PHYSICAL core, precomputed transposed
    restriction. Both the `--impl reference` arm and the `cpu_baseline` of the GPU arm time exactly this object and report
    the median step, so the two CPU numbers of one record agree."""

    def __init__(self, prob, sample_elems=0):
        from oracle import pyoracle as O

        self.native = O.use_native_build()  # -march=native on this host (falls back to the portable prebuilt library)
        self.O = O
        nd = prob["nd"]
        p, q1d = prob["p"], prob["q1d"]
        self.ne = prob["mesh"].ne
        self.ns = self.ne if sample_elems <= 0 else min(self.ne, sample_elems)
        self.interp, self.curl, _ = O.nd_hex_tables(p, q1d)
        idx, ori = nd.native_restriction()
        self.idx, self.ori = np.ascontiguousarray(idx[: self.ns]), np.ascontiguousarray(ori[: self.ns])
        self.qd = O.geom_hex_qdata(prob["xe"][: self.ns], prob["mesh"].attr[: self.ns], prob["mesh_order"], q1d)
        self.blob = prob["blob"]
        self.x = np.random.default_rng(1).random(nd.ndofs)
        self.y = np.zeros(nd.ndofs)
        self.ndofs = nd.ndofs
        self.physical = O.physical_cores()
        self.quota = cpu_quota()
        nthreads = self.physical if self.quota is None else max(1, min(self.physical, int(self.quota)))
        self.arm = O.BlockedApply(O.CURLCURL_MASS, self.interp, self.curl, self.idx, self.ori, self.qd, self.blob, nd.ndofs, nthreads=nthreads)
        self.cores = self.arm.threads  # pinned threads, one per physical core, at most the container's CPU quota
        self.logical = os.cpu_count() or 1

    def step(self):
        self.y[:] = 0.0
        t0 = time.perf_counter()
        self.arm.apply_add(self.x, self.y)
        return time.perf_counter() - t0

    def median_step(self, steps, warmup=2):
        for _ in range(max(1, warmup)):
            self.step()
        dts = sorted(self.step() for _ in range(max(1, steps)))
        return dts[len(dts) // 2], dts

    @property
    def dofs_per_step(self):
        return self.ndofs * (self.ns / self.ne)

    def describe(self, steps):
        return (f"{self.ns} of {self.ne} elements per step, median of {steps} steps; dense non-tensor basis apply (oracle port of the libCEED "
                f"/cpu/self path, blocks of 8 elements, {self.cores} threads pinned one per physical core; host: {self.physical} physical cores / "
                f"{self.logical} logical CPUs, container CPU quota {'none' if self.quota is None else round(self.quota, 1)}, "
                f"{'-march=native build on this host' if self.native else 'portable x86-64-v3 build'}; the reference itself is unbuildable here)")


def run_reference(args, rank, world):
    if rank != 0:
        return
    prob = build_problem(args.n, args.order, args.warp, coefficient=args.coefficient)
    ref = CpuReference(prob, args.cpu_sample_elems)  # default: the whole 2M-dof mesh every step
    steps = max(1, args.steps)
    med, dts = ref.median_step(steps, warmup=max(1, min(args.warmup, 3)))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ref.y, 0, 1)
    value = float(ref.dofs_per_step / med / 1e6)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, prob, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": ref.describe(steps),
                         "min_ms": 1e3 * dts[0], "max_ms": 1e3 * dts[-1]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, prob, world):
    nd = prob["nd"]
    return {
        "workload": f"ND hex p={args.order} curl-curl+mass ParOperator Mult (P, local apply, P^T) on a uniform {args.n}^3-elements-per-GPU box mesh, stored per-point geometry"
                    + (" (assembled D)" if args.assemble_qdata else " (J^-T, w detJ; coefficient applied on the fly)")
                    + ("; four striped materials with full 3x3 tensors" if args.coefficient == "matrix4" else "; one isotropic material")
                    + (f"; mesh warped by {args.warp}" if args.warp else ""),
        "order": args.order, "elements_per_gpu": int(args.n ** 3), "global_true_dofs": int(nd.ndofs), "n_gpus": world,
        "partition": ("1 block per GPU; shared dofs exchanged through peer memory over NVLink (CUDA-IPC mailboxes: stores + epoch flags, "
                      "fused into one kernel before and one after the element kernel, replayed from a CUDA graph)"
                      if os.environ.get("B2P_HALO_P2P", "1") == "1" else
                      "1 block per GPU; shared dofs exchanged by NCCL grouped send/recv") if world > 1 else "single partition",
        "vector": "true-dof (T) vector",
        "l2_policy": "L2 flushed (256 MiB write" + (", then read back" if os.environ.get("B2P_BENCH_FLUSH", "write") == "write_read" else "") + ") between timed iterations",
    }


def run_experiments(args):
    """Side measurements of the same run, each taken by a child process (a failure or hang of one of them cannot touch the
    headline numbers) and printed as ITS OWN short JSON line -- {"experiment": name, ...} -- before the headline line, so that
    none of them can fall off a log tail. The headline line stays the last line of the output."""
    # no experiment STARTS after budget_s; each is cut off at 150 s, so the side measurements end within ~7 minutes in the worst case
    # (they took 1.5 minutes on B200 with the round-2 list of 13, profiles/r02_bench_n1_with_experiments.jsonl)
    t_start, budget_s = time.time(), float(os.environ.get("B2P_BENCH_EXPERIMENT_BUDGET_S", "270"))
    common = ["--steps", str(args.steps), "--warmup", str(args.warmup), "--order", str(args.order), "--n", str(args.n),
              "--no-cpu-baseline", "--no-experiments"]
    # (1) the same bench on other kernels / coefficients: value, kernel time and roofline fraction of each
    variants = {
        "matrix_coefficient_warped_mesh": (["--coefficient", "matrix4", "--warp", "0.05"], {}),
        "round1_kernel_nd_hex_apply4": ([], {"B2P_ND_KERNEL": "4"}),
        "without_pdl_zero_fill_overlap": ([], {"B2P_PDL": "0"}),
        "l2_flush_written_then_read_back": ([], {"B2P_BENCH_FLUSH": "write_read"}),
    }
    if args.order == 3:
        # the high-order kernel (nd_hex_apply7_kernel: CTA per element batch) at about the same number of dofs
        variants.update({
            "hex_order4_2p4M_dofs": (["--order", "4", "--n", "23"], {}),
            "hex_order5_2p2M_dofs": (["--order", "5", "--n", "18"], {}),
            "hex_order6_2p2M_dofs": (["--order", "6", "--n", "15"], {}),
        })
    # (2) prepared tool measurements (tools/): one JSON line each
    tools = {
        "complex_fused_and_pair_apply": (["tools/zfused_bench.py", "--steps", "50"], {}),
        "solver_loop_p3_2M": (["tools/solver_bench.py"], {}),
        "cylinder_cavity_p4_vs_reference_eig_csv": (["tools/cylinder_bench.py", "--order", "4", "--refine", "0", "--nev", "4"], {}),
        "tet_dense_p3_1M_dofs": (["tools/tet_bench.py", "--order", "3", "--n", "21", "--steps", "20", "--terms"], {}),
        "tet_dense_p6_1M_dofs": (["tools/tet_bench.py", "--order", "6", "--n", "11", "--steps", "10"], {}),
        # BASELINE config 3's workflow in miniature on one GPU: frequency sweep on order-3 tets, operators re-coefficiented in
        # place, SetOperators of the p-multigrid per frequency, complex FGMRES + real V-cycle (PCMatReal)
        "driven_sweep_tets_p3": (["tools/driven_sweep_bench.py", "--order", "3", "--n", "12", "--freqs", "4"], {}),
        # BASELINE config 2 at size: cylinder cavity, ND order 4, p-multigrid {1, 2, 4}, Chebyshev order 8 + Hiptmair, 7.94M dofs
        "cylinder_cavity_p4_7p9M_dofs": (["tools/cylinder_bench.py", "--order", "4", "--refine", "3", "--nev", "2", "--tol", "1e-8",
                                          "--coarse-tol", "1e-4"], {"B2P_COARSE_ASSEMBLED": "1"}),
    }
    child = os.environ.get("B2P_BENCH_CHILD")  # (the CPU dry-run harness points this at itself)
    if child:  # CPU dry run: tiny sizes
        tools = {"complex_fused_and_pair_apply": (["tools/zfused_bench.py", "--n", "3", "--steps", "2"], {}),
                 "solver_loop_p3_2M": (["tools/solver_bench.py", "--n", "3"], {})}

    def emit(name, payload):
        print(json.dumps(dict({"experiment": name}, **payload)), flush=True)

    for name, (extra, env) in variants.items():
        if time.time() - t_start > budget_s:
            emit(name, {"skipped": "experiment time budget used up"})
            continue
        try:
            r = subprocess.run([sys.executable, child or os.path.abspath(__file__)] + common + extra,
                               env=dict(os.environ, B2P_BENCH_EXPERIMENTS="0", **env), capture_output=True, text=True, timeout=150)
            last = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
            if not last:
                raise RuntimeError("no result line; stderr tail: " + r.stderr.strip()[-160:])
            d = json.loads(last[-1])
            emit(name, {"args": extra, "env": env, "value": d["value"], "unit": d["unit"], "ms_per_step": d["ms_per_step"],
                        "kernel": d["roofline"]["kernel"], "kernel_ms": d["roofline"]["kernel_ms"], "roofline_frac": d["roofline"]["frac"]})
        except Exception as exc:
            emit(name, {"args": extra, "env": env, "failed": f"{type(exc).__name__}: {str(exc)[:200]}"})
    for name, (cmd, env) in tools.items():
        if time.time() - t_start > budget_s:
            emit(name, {"skipped": "experiment time budget used up"})
            continue
        try:
            argv = [sys.executable] + ([child] if child else []) + [os.path.join(ROOT, cmd[0])] + cmd[1:]
            r = subprocess.run(argv, env=dict(os.environ, B2P_BENCH_EXPERIMENTS="0", **env), capture_output=True, text=True, timeout=150, cwd=ROOT)
            last = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
            if not last:
                raise RuntimeError("no result line; stderr tail: " + r.stderr.strip()[-160:])
            emit(name, json.loads(last[-1]))
        except Exception as exc:
            emit(name, {"failed": f"{type(exc).__name__}: {str(exc)[:200]}"})


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from palace_b200 import capi

    assert torch.cuda.is_available(), "bench.py needs a GPU (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    parts = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}.get(world)
    assert parts is not None, "--gpus must be 1, 2, 4 or 8"
    if world > 1:
        # one NCCL communicator inside the library (unique id from rank 0, shipped over torch.distributed)
        uid = [capi.Ctx.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx = capi.Ctx(local_rank, nccl_uid=uid[0], rank=rank, nranks=world)
    else:
        ctx = capi.Ctx(local_rank)
    capi.set_stream(ctx)

    # weak scaling: an (n*px, n*py, n*pz) box split into px*py*pz blocks of n^3 elements, one per GPU
    from palace_b200.host import hexmesh as hm
    from palace_b200.host import partition as pt

    gn = (args.n * parts[0], args.n * parts[1], args.n * parts[2])
    prob = build_problem(gn, args.order, args.warp, size=(float(parts[0]), float(parts[1]), float(parts[2])), coefficient=args.coefficient)
    p, q1d = prob["p"], prob["q1d"]
    gnd = prob["nd"]
    if world > 1:
        elem_rank = hm.partition_box(gn, parts)
        ls = pt.partition_space(gnd, elem_rank, rank, world, order=pt.interface_order(prob["mesh"].elems, elem_rank, rank))
        nd, elems = ls.space, ls.elems
        halo = capi.Halo(ctx, ls.n_true, ls.n_ghost, ls.nbr, ls.send_counts, ls.send_idx, ls.recv_counts)
        n_true, lsize = ls.n_true, ls.lsize
        if os.environ.get("B2P_HALO_P2P", "1") == "1":  # NVLink peer-memory exchange instead of NCCL send/recv
            def gather(blob):
                out = [None] * world
                dist.all_gather_object(out, blob)
                return out
            halo.enable_p2p(gather)
    else:
        nd, elems, halo = gnd, np.arange(prob["mesh"].ne), None
        n_true = lsize = gnd.ndofs
    N_global = gnd.ndofs
    geom = capi.Geom.hex(ctx, prob["xe"][elems], prob["mesh"].attr[elems], prob["mesh_order"], q1d, prob["nB"], prob["nG"],
                         prob["tabs"].qw)
    idx, ori = nd.native_restriction()
    t = prob["tabs"]
    op = capi.Op.create(ctx, geom, capi.CURLCURL_MASS, p, lsize, idx, ori, nd.dof_map, t.Bo, t.Bc, t.Gc, prob["blob"],
                        assemble=bool(args.assemble_qdata))
    A = capi.Operator.par(ctx, n_true, lsize, [op], None, None, diag_policy=1, halo=halo)
    if world > 1:
        A.set_interior(ls.n_interior)  # interior elements first: the kernel waits for ghosts only when it reaches the interface

    prob["local_ne"] = int(elems.size)
    prob["local_dofs"] = int(lsize)
    N = n_true
    xh = torch.from_numpy(np.random.default_rng(1 + rank).random(N)).pin_memory()
    yh = torch.empty(N, dtype=torch.float64).pin_memory()
    xd = xh.cuda()
    yd = torch.empty_like(xd)
    xl = torch.zeros(lsize, dtype=torch.float64, device="cuda")
    yl = torch.zeros(lsize, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()

    qbytes = prob["local_ne"] * 10 * q1d ** 3 * 8
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")  # > 126 MB L2
    # B2P_BENCH_FLUSH=write_read (side experiment only): read the buffer back after writing it, so the 126 MB the flush
    # leaves in L2 are CLEAN lines -- a plain write leaves them dirty and the timed kernels pay their write-back.
    flush_read = os.environ.get("B2P_BENCH_FLUSH", "write") == "write_read"

    def do_flush():
        flush.zero_()
        if flush_read:
            torch.sum(flush)

    def step_device():
        A.mult(xd, yd)  # ParOperator::Mult: P (halo), zero-fill, local apply, P^T (halo)

    def step_e2e():
        xd.copy_(xh, non_blocking=True)
        A.mult(xd, yd)
        yh.copy_(yd, non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step_device()
    barrier()

    # ---- device-resident timing (value): CUDA events per step, L2 flushed between steps if needed ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_wall0 = time.time()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        if flush is not None:
            do_flush()
        a.record(stream)
        step_device()
        b.record(stream)
    barrier()
    t_wall1 = time.time()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, yd.cpu().numpy(), rank, world)
    ms = np.array([a.elapsed_time(b) for a, b in evs])
    total_ms = float(ms.sum())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    tt = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    value = N_global * args.steps / (total_ms * 1e-3) / 1e6

    # ---- kernel-only timing for the roofline (memset excluded) ----
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(args.steps, 50))]
    for a, b in kev:
        yl.zero_()
        if flush is not None:
            do_flush()
        a.record(stream)
        op.apply_add(xl, yl)  # the local element kernel alone, all elements of this rank
        b.record(stream)
    torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    abytes = op.algorithmic_bytes()
    # which sum-factorised kernel the library dispatches for this operator (b2p_core.cu:apply_range)
    forced = os.environ.get("B2P_ND_KERNEL", "0")
    kernel_name = "nd_hex_apply4_kernel"
    if forced in ("0", "6") and args.order in (2, 3) and not args.assemble_qdata:
        kernel_name = "nd_hex_apply6_kernel"
    elif forced in ("0", "7") and args.order in (4, 5, 6) and not args.assemble_qdata:
        kernel_name = "nd_hex_apply7_kernel"
    traffic = None
    try:  # DRAM bytes of the same kernel/launch shape from the committed ncu capture (profiles/)
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)
        if args.order == 3 and args.n == 29 and not args.assemble_qdata and world == 1:
            k = tr[kernel_name + "<3,4,CURLCURL_MASS,geom>"]
            traffic = k["dram_bytes_read"] + k["dram_bytes_write"]
    except Exception:
        pass
    peak, peak_src = measured_peak_gbs()
    achieved = abytes / (k_ms * 1e-3) / 1e9

    # ---- end to end through the C ABI with host buffers ----
    # serial (latency of one call): pinned host x -> device, Mult, device y -> pinned host, on one stream
    for _ in range(3):
        step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = min(args.steps, 50)
    e0.record(stream)
    for _ in range(e2e_steps):
        step_e2e()
    e1.record(stream)
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_serial = N_global * e2e_steps / (float(te.item()) * 1e-3) / 1e6
    e2e_value, e2e_mode = e2e_serial, "serial: H2D, Mult, D2H on one stream"
    if world == 1 and os.environ.get("B2P_E2E_PIPELINE", "1") == "1":
        try:
            # throughput of independent calls: double-buffered device vectors on three streams, so the H2D copy of
            # step k+1 and the D2H copy of step k-1 (opposite PCIe directions) overlap the Mult of step k. Every
            # step still copies its own x from pinned host memory and its own y back inside the timed region.
            s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
            xb = [torch.empty_like(xd) for _ in range(2)]
            yb = [torch.empty_like(yd) for _ in range(2)]
            yhb = [torch.empty(N, dtype=torch.float64).pin_memory() for _ in range(2)]
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_cmp = [torch.cuda.Event() for _ in range(2)]
            ev_out = [torch.cuda.Event() for _ in range(2)]
            capi.set_stream(ctx, s_cmp.cuda_stream)

            def step_pipe(k):
                b = k & 1
                with torch.cuda.stream(s_in):
                    if k >= 2:
                        s_in.wait_event(ev_cmp[b])  # Mult k-2 has consumed xb[b]
                    xb[b].copy_(xh, non_blocking=True)
                    ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    if k >= 2:
                        s_cmp.wait_event(ev_out[b])  # yb[b] of step k-2 has been copied out
                    A.mult(xb[b], yb[b])  # enqueued on the context stream (= s_cmp)
                    ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    yhb[b].copy_(yb[b], non_blocking=True)
                    ev_out[b].record(s_out)

            for k in range(4):
                step_pipe(k)
            barrier()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record(s_in)
            for k in range(e2e_steps):
                step_pipe(k)
            p1.record(s_out)  # after the last D2H copy
            barrier()
            capi.set_stream(ctx, stream.cuda_stream)
            # same x every step: the pipelined result must equal the serial one (up to the order of the scatter-adds)
            ok = bool(torch.allclose(yhb[(e2e_steps - 1) & 1], yh, rtol=1e-11, atol=1e-13))
            if ok:
                e2e_value = N_global * e2e_steps / (p0.elapsed_time(p1) * 1e-3) / 1e6
                e2e_mode = "pipelined: double-buffered, H2D(k+1) and D2H(k-1) overlap Mult(k) on three streams"
            else:
                e2e_mode += " (pipelined result mismatch: not reported)"
        except Exception as exc:  # never lose the bench line to the optional pipelined leg
            try:
                torch.cuda.synchronize()
                capi.set_stream(ctx, stream.cuda_stream)
            except Exception:
                pass
            e2e_value, e2e_mode = e2e_serial, f"serial: H2D, Mult, D2H on one stream (pipelined leg failed: {type(exc).__name__}: {exc})"

    # ---- N > 1: parity of the partitioned Mult inside the recorded run (outside every timed region) ----
    # Every rank applies the distributed operator to its slice of ONE global vector; rank 0 applies the single-partition
    # operator of the whole mesh to the same vector and compares on each rank's owned dofs (the reference checks partition
    # independence by running its regression suite at several rank counts).
    partition_parity = None
    if world > 1:
        xg = np.random.default_rng(12345).standard_normal(N_global)
        own = ls.local_to_global[: ls.n_true]
        xp = torch.from_numpy(np.ascontiguousarray(xg[own])).cuda()
        yp = torch.empty_like(xp)
        A.mult(xp, yp)
        torch.cuda.synchronize()
        pieces = [None] * world if rank == 0 else None
        dist.gather_object((np.asarray(own), yp.cpu().numpy()), pieces, dst=0)
        if rank == 0:
            try:
                geom_g = capi.Geom.hex(ctx, prob["xe"], prob["mesh"].attr, prob["mesh_order"], q1d, prob["nB"], prob["nG"], prob["tabs"].qw)
                gi, go = gnd.native_restriction()
                op_g = capi.Op.create(ctx, geom_g, capi.CURLCURL_MASS, p, gnd.ndofs, gi, go, gnd.dof_map, t.Bo, t.Bc, t.Gc, prob["blob"],
                                      assemble=bool(args.assemble_qdata))
                A_g = capi.Operator.par(ctx, gnd.ndofs, gnd.ndofs, [op_g], None, None, diag_policy=1, halo=None)
                xgd = torch.from_numpy(xg).cuda()
                ygd = torch.empty_like(xgd)
                A_g.mult(xgd, ygd)
                torch.cuda.synchronize()
                y_ref = ygd.cpu().numpy()
                err = max(float(np.abs(yv - y_ref[o]).max()) for o, yv in pieces) / float(np.abs(y_ref).max())
                covered = int(sum(o.size for o, _ in pieces))
                partition_parity = {"max_rel_err": err, "dofs_checked": covered, "ok": bool(err < 1e-12 and covered == N_global),
                                    "against": "single-partition ParOperator::Mult of the whole mesh on rank 0, same global vector"}
                del A_g, op_g, geom_g, xgd, ygd
            except Exception as exc:
                partition_parity = {"failed": f"{type(exc).__name__}: {str(exc)[:200]}"}

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, prob, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(N_global * 8), "d2h_bytes_per_step": int(N_global * 8),
                    "mode": e2e_mode, "serial_value": e2e_serial},
            # kernels of this library per rank and timed step: N = 1: zero_release_kernel + the element kernel (the zero-fill is a
            # cudaMemset, not a kernel of ours, with B2P_PDL=0); N > 1: p2p_pre_kernel + element kernel + p2p_post_kernel
            "gpu_launches": int(args.steps * (3 if world > 1 else (1 if os.environ.get("B2P_PDL", "1") == "0" else 2))),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": kernel_name, "kernel_ms": k_ms,
                         "algorithmic_bytes_per_launch": int(abytes)},
        }
        if partition_parity is not None:
            line["partition_parity"] = partition_parity
        if not args.no_cpu_baseline:
            base_prob = prob if world == 1 else build_problem(args.n, args.order, args.warp, coefficient=args.coefficient)
            ref = CpuReference(base_prob, args.cpu_sample_elems)
            med, dts = ref.median_step(10, warmup=2)
            line["cpu_baseline"] = {"value": ref.dofs_per_step / med / 1e6, "unit": UNIT, "cores": ref.cores, "kind": "port",
                                    "sample": ref.describe(10), "min_ms": 1e3 * dts[0], "max_ms": 1e3 * dts[-1]}
        if world == 1 and not args.no_experiments and os.environ.get("B2P_BENCH_EXPERIMENTS", "1") == "1":
            run_experiments(args)  # one JSON line each, before the headline
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
