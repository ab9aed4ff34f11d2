#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU kd-tree on the host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...      # one rank per GPU, weak scaling
    python bench.py ... --dump-outputs DIR                     # + the last timed step's radii as DIR/radius.npy
                                                               #   (rank 0's only: other ranks' batches are not written)

A step = one pass of the hot path over one batch: `pc_radius_batch` (safeRegionRrtStar::radiusSearch,
Planner/src/corridor_finder.cpp:113-133) for a batch of RRT* sample points against the resident index of the
C2 map (1M-point synthetic forest, clean_demo parameters).  `value` = queries/s with the batch resident in
HBM; `e2e` = the same call with pinned HOST buffers (H2D + D2H inside the timed region).  One JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "exact NN radius queries/s on 1M-pt cloud"
UNIT = "queries/s"
N_POINTS = 1_000_000
CLOUD_SEED = 1
PARAMS = dict(search_margin=0.25, max_radius=1.5, sample_range=30.0)   # clean_demo.launch:31-34
BYTES_PER_QUERY = 16            # algorithmic: 12 B query (xyz float32) in + 4 B radius out
FRAME_POINTS = 300_000          # C3 frame for the build-ms metric
# ncu figures of ONE launch of the dominant kernel on the default workload (dram bytes, warp instructions) live in
# profiles/ncu_dominant_kernel.json, written by `scripts/ncu_summary.py traffic` from an `ncu --set full` capture together
# with a hash of the kernel sources it was taken on; figures taken on other sources are reported as stale (null)
NCU_FILE = os.path.join(ROOT, "profiles", "ncu_dominant_kernel.json")
KERNEL_SOURCES = ["common.cuh", "lbvh.cuh", "build_kernels.cuh", "query_kernels.cuh", "radix_sort.cuh"]


def kernel_source_hash():
    import hashlib
    h = hashlib.sha1()
    for f in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "pointcloudtraj_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def ncu_figures(queries):
    """-> (dict or None, note): the committed ncu figures if they were captured on the current kernel sources and batch size."""
    try:
        d = json.load(open(NCU_FILE))
    except Exception:
        return None, "profiles/ncu_dominant_kernel.json missing"
    if d.get("source_sha1") != kernel_source_hash():
        return None, f"stale: captured at commit {d.get('commit')} on other kernel sources"
    if int(d.get("queries", 0)) != int(queries):
        return None, f"captured for {d.get('queries')} queries per launch"
    return d, f"profiles/{d.get('summary_file')} (ncu --set full at commit {d.get('commit')}, per launch)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--queries", type=int, default=10_000_000, help="queries per step per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=1_000_000)
    ap.add_argument("--ref-sample", type=int, default=200_000, help="queries per step of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the radii the last timed step returned to DIR/radius.npy; "
                         "with several ranks only rank 0's radii are written, not the other ranks' batches")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# --dump-outputs writes at most this many bytes; a larger output is thinned to every k-th value (k fixed by its size)
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, radius):
    """Write the last timed step's radii as out_dir/radius.npy, so that two builds can be compared value for value."""
    stride = -(-radius.nbytes // DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "radius.npy"), np.ascontiguousarray(radius[::stride]))


def workload_config(args):
    """Identical in both arms (the driver compares them)."""
    return {"workload": "C2: 1M-point synthetic forest map (jittered lattice, seed 1), radiusSearch batches of "
                        f"{args.queries} uniform in-box RRT* samples per GPU, clean_demo params "
                        "(search_margin 0.25, max_radius 1.5, sample_range 30)",
            "points": N_POINTS, "queries_per_step_per_gpu": args.queries,
            "l2_policy": "inputs+outputs per step (16 B/query x 1e7 = 160 MB) exceed the 126 MB L2"}


def host_threads():
    """All the host threads this process may use -- NOT OMP_NUM_THREADS, which torch.distributed.run sets to 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def make_cloud():
    from pointcloudtraj_b200 import synth
    return synth.forest_cloud(N_POINTS, seed=CLOUD_SEED, variant="J", return_half=True)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons, streamed every 50 ms while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc = gpu, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        time.sleep(0.3)          # let the first samples arrive before the timed region starts

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            rows = [[c.strip() for c in ln.split(",")] for ln in out.splitlines() if ln.strip()]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(rows)}


# ---- CPU legs (the only places that execute oracle/) --------------------------------------------------
def cpu_reference_tree(pts):
    import oracle
    order = np.random.default_rng(0).permutation(len(pts))
    if oracle.have_reference():
        return oracle.KdReference().build(pts, order), "reference"
    return oracle.KdOracle().build(pts, order), "port"


def cpu_radius(tree, kind, q, start):
    import oracle
    P = oracle.RadiusParams.make(start=start, **PARAMS)
    if kind == "reference":
        return tree.radius_batch(P, q, nthreads=host_threads())
    return tree.radius_batch(P, q)[0]


def cpu_baseline(pts, q, start, sample):
    import oracle
    t0 = time.perf_counter()
    tree, kind = cpu_reference_tree(pts)
    t_build = time.perf_counter() - t0
    qs = q[:sample]
    t0 = time.perf_counter()
    r = cpu_radius(tree, kind, qs, start)
    dt = time.perf_counter() - t0
    cores = host_threads() if kind == "reference" else 1
    return {"value": len(qs) / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"first {len(qs)} queries of the step batch on the same 1M-point cloud "
                      f"(kd_insert3 build {t_build * 1e3:.0f} ms single-threaded, not included)",
            "build_ms": t_build * 1e3}, r


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pointcloudtraj_b200 import synth
    pts, half = make_cloud()
    start = (0.0, 0.0, 2.0)
    tree, kind = cpu_reference_tree(pts)
    cores = host_threads() if kind == "reference" else 1
    if kind == "reference" and (os.cpu_count() or 1) > 1 and cores <= 1:
        print("[bench] WARNING: the reference arm sees one host thread (restricted CPU affinity)", file=sys.stderr)
    m = args.ref_sample
    qs = [synth.rrt_queries(m, half, seed=100 + s) for s in range(args.warmup + args.steps)]
    for s in range(args.warmup):
        cpu_radius(tree, kind, qs[s], start)
    t0 = time.perf_counter()
    for s in range(args.steps):
        r_last = cpu_radius(tree, kind, qs[args.warmup + s], start)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r_last)
    val = m * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "reference_step_sample": m,
                             "host_cpus": os.cpu_count(), "omp_num_threads_env_ignored": os.environ.get("OMP_NUM_THREADS"),
                             "sample": f"{m} queries per step (bounded sample of the {args.queries}-query batch), "
                                       "kd_nearest3 + radiusSearch epilogue, OpenMP over queries"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---- this repo's arm -----------------------------------------------------------------------------------
def bind_to_gpu_numa_node(props):
    """Multi-GPU runs: pin this rank's threads to the CPUs next to its GPU (NVML's ideal CPU affinity) BEFORE any pinned
    host buffer is allocated, so that the e2e leg's DMA traffic stays on the GPU's own socket (first-touch allocation).
    Returns the CPU list (for the JSON line) or None when NVML gives no answer."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus_id = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus_id.encode())
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception as e:  # noqa: BLE001 -- binding is an optimisation only
        print(f"[bench] NUMA binding skipped: {e}", file=sys.stderr)
    return None


def run_b200(args):
    import torch
    import torch.distributed as dist
    from pointcloudtraj_b200 import PC_DEVICE, PcRadiusParams, PointCloudIndex, synth  # noqa: F401

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa_node(torch.cuda.get_device_properties(local)) if world > 1 else None
    # one explicit non-default stream for everything: the library's kernels, torch's copies and the timing events
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    M = args.queries
    start = (0.0, 0.0, 2.0)

    # the cloud lives on rank 0 only: rank 0 builds the index, ONE ncclBroadcast (pc_index_broadcast) replicates the
    # built index into every rank's handle; after that no collective is on the data path
    stream = torch.cuda.current_stream().cuda_stream
    ix = PointCloudIndex(max_points=N_POINTS, device=local, stream=stream)
    meta = torch.zeros(1, dtype=torch.float64, device=dev)
    build_ms = []
    t_pts = None
    if rank == 0:
        pts, half = make_cloud()
        t_pts = torch.from_numpy(pts).to(dev)
        meta[0] = half
        for _ in range(5):
            ix.build(t_pts)
            build_ms.append(ix.last_build_ms())
    bcast_ms = 0.0
    if world > 1:
        from pointcloudtraj_b200.dist import Replicator
        rep = Replicator(rank, world, local)
        dist.broadcast(meta, 0)
        rep.broadcast(ix, 0)                      # warm-up (NCCL channel setup)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        rep.broadcast(ix, 0)
        e1.record()
        torch.cuda.synchronize()
        bcast_ms = e0.elapsed_time(e1)
        assert ix.size == N_POINTS
    half = float(meta.item())
    replica_ok = None
    if world > 1:
        # every rank answers the same probe batch against its replica; all answers must equal rank 0's
        probe = torch.from_numpy(synth.rrt_queries(200_000, half, seed=7)).to(dev)
        pi, pd = ix.nearest(probe)
        ref_i, ref_d = pi.clone(), pd.clone()
        dist.broadcast(ref_i, 0)
        dist.broadcast(ref_d, 0)
        ok = torch.tensor([int(bool((pi == ref_i).all().item() and (pd == ref_d).all().item()))], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        replica_ok = bool(ok.item())
    P = PcRadiusParams.make(start=start, **PARAMS)

    # per-rank query batch (weak scaling: every GPU answers its own M queries per step)
    q_host = synth.rrt_queries(M, half, seed=1000 + rank)
    # share of the batch that radiusSearch answers without a cloud query (farther than sample_range + max_radius from start)
    early_frac = float((np.sqrt(((q_host.astype(np.float64) - np.array(start)) ** 2).sum(1)) > PARAMS["sample_range"] + PARAMS["max_radius"]).mean())
    q_pin = torch.from_numpy(q_host).pin_memory()
    t_q = q_pin.to(dev, non_blocking=True)
    t_r = torch.empty(M, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    import ctypes as C
    lib = ix._L

    t_rs = [t_r, torch.empty_like(t_r), torch.empty_like(t_r)]

    def step_device(space=PC_DEVICE, k=0):
        # PC_DEVICE: on the handle's stream.  PC_DEVICE_ASYNC (3): batches rotate over the library's three internal streams,
        # so one batch's ordering pass overlaps the previous batch's search; every batch in flight has its own output buffer.
        rc = lib.pc_radius_batch(ix._h, C.c_void_p(t_q.data_ptr()), M, 3, space, 0, C.byref(P), C.c_void_p(t_rs[k % 3].data_ptr()), None)
        if rc != 0:
            raise RuntimeError(lib.pc_last_error(ix._h).decode())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ix.profile(True)
    for k in range(args.warmup):
        step_device(3, k)
    ix.sync()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ix.launches(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    search_ms, order_ms = [], []
    e0.record()
    for k in range(args.steps):
        step_device(3, k)
    ix.sync()                 # all internal streams done; e1 is recorded after the last batch has finished
    e1.record()
    barrier()
    launches = ix.launches()
    elapsed_ms = e0.elapsed_time(e1)
    # step k wrote t_rs[k % 3]; the loops below overwrite these buffers, so the last timed step's radii are copied out now
    r_last = t_rs[(args.steps - 1) % 3].cpu().numpy() if args.dump_outputs and rank == 0 else None
    # kernel-level durations of the dominant kernel, measured with CUDA events around it (separate short loop so
    # that reading the events does not stall the timed region above)
    for _ in range(min(args.steps, 10)):
        step_device()
        a, b = ix.last_batch_ms()
        order_ms.append(a)
        search_ms.append(b)
    ix.profile(False)
    # the same batch with the sensing-range early-out disabled (sample_range < 0): every query is searched
    P_all = PcRadiusParams.make(start=start, search_margin=PARAMS["search_margin"], max_radius=PARAMS["max_radius"], sample_range=-1.0)
    t_all = torch.empty_like(t_r)

    def step_all():
        rc = lib.pc_radius_batch(ix._h, C.c_void_p(t_q.data_ptr()), M, 3, PC_DEVICE, 0, C.byref(P_all), C.c_void_p(t_all.data_ptr()), None)
        if rc != 0:
            raise RuntimeError(lib.pc_last_error(ix._h).decode())

    for _ in range(2):
        step_all()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    for _ in range(5):
        step_all()
    eb.record()
    torch.cuda.synchronize()
    all_searched_qps = M * 5 / (ea.elapsed_time(eb) * 1e-3)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = world * M * args.steps / (elapsed_ms * 1e-3)

    # e2e: the same call through the C ABI with pinned HOST buffers; every step copies its 120 MB batch host->device and its
    # 40 MB of radii device->host inside the timed region.
    #  (a) one blocking PC_HOST call per step (internally a chunked 3-stream pipeline): the latency a single caller sees;
    #  (b) PC_HOST_ASYNC: the steps are enqueued back to back on three internal streams (each step's batch in its own
    #      output buffer) and waited for once -- consecutive steps overlap their PCIe copies with each other's kernels.
    #      This is the throughput a planner that double-buffers its sample batches gets, and the reported e2e value.
    r_pins = [torch.empty(M, dtype=torch.float32).pin_memory() for _ in range(3)]
    qp = q_pin.numpy()
    rps = [r.numpy() for r in r_pins]

    def step_host(space, k=0):
        rc = lib.pc_radius_batch(ix._h, C.c_void_p(qp.ctypes.data), M, 3, space, 0, C.byref(P), C.c_void_p(rps[k % 3].ctypes.data), None)
        if rc != 0:
            raise RuntimeError(lib.pc_last_error(ix._h).decode())

    def max_over_ranks(seconds):
        t = torch.tensor([seconds], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e2e_steps = max(3, min(args.steps, 12))
    for _ in range(2):
        step_host(0)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host(0)
    torch.cuda.synchronize()
    e2e_blocking = world * M * e2e_steps / max_over_ranks(time.perf_counter() - t0)
    for k in range(3):
        step_host(2, k)
    ix.sync()
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        step_host(2, k)
    ix.sync()
    e2e_val = world * M * e2e_steps / max_over_ranks(time.perf_counter() - t0)
    same = all(bool((r.to(dev) == t_r).all().item()) for r in r_pins)
    clocks = sampler.stop() if sampler else None     # sampled across the device-timed and the end-to-end regions

    # host roof of the buffer API: what the host side of the PCIe fabric delivers when every rank moves one step's bytes
    # (12 B/query in, 4 B/query out, pinned memory, both directions at once) with NO kernel in between
    cp_in, cp_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_q2, d_r2 = torch.empty_like(t_q), torch.empty_like(t_r)

    def copy_step():
        with torch.cuda.stream(cp_in):
            d_q2.copy_(q_pin, non_blocking=True)
        with torch.cuda.stream(cp_out):
            r_pins[0].copy_(d_r2, non_blocking=True)

    for _ in range(2):
        copy_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        copy_step()
    torch.cuda.synchronize()
    host_roof_s = max_over_ranks(time.perf_counter() - t0)
    host_roof_gbs = world * 16 * M * e2e_steps / host_roof_s / 1e9
    del d_q2, d_r2

    # device-generated path (pc_expand_batch): a step's M samples are drawn on the device from the planner's engine state
    # (minstd_rand0 + libstdc++'s uniform_real_distribution, bit-identical with genSample), steered from their nearest vertex of a
    # frozen node set, answered by radiusSearch, and only the candidates the expansion loop keeps come back -- no 12 B/query
    # H2D.  Timed by the host clock around the C-ABI call (host buffers in, host buffers out), like e2e.
    from pointcloudtraj_b200 import PcSampler
    rngn = np.random.default_rng(77 + rank)
    n_nodes = 4096
    node_coord = np.column_stack([rngn.uniform(-25, 25, n_nodes), rngn.uniform(-25, 25, n_nodes), rngn.uniform(0.7, 4.0, n_nodes)])
    node_coord[0] = start
    node_radius = rngn.uniform(0.6, 1.25, n_nodes).astype(np.float32)
    node_valid = np.ones(n_nodes, np.uint8)
    smp = PcSampler.make(start, (0.8 * half, 0.5 * half, 2.0), (-half, half, -half, half, 0.0, 4.0), PARAMS["sample_range"], 0.6, 0.3, 0.1,
                         engine_state=1 + rank)
    dg = None
    with PointCloudIndex(max_points=1 << 16, device=local, stream=stream) as nodes_ix:
        from pointcloudtraj_b200 import _lib as pclib
        nset = pclib.PcNodeSet(n_nodes, node_coord.ctypes.data, node_radius.ctypes.data, node_valid.ctypes.data)
        cand_pin = torch.empty(32 * M, dtype=torch.uint8).pin_memory()         # pc_candidate records, pinned like the e2e buffers
        cand_np = cand_pin.numpy()
        cnt_c, st_c = C.c_int64(0), C.c_uint32(0)

        def step_expand(k):
            rc = lib.pc_expand_batch(ix._h, nodes_ix._h, C.byref(nset), C.byref(smp), C.byref(P), 0.0, 0.6, k, C.c_void_p(cand_np.ctypes.data), M,
                                     C.byref(cnt_c), C.byref(st_c))
            if rc != 0:
                raise RuntimeError(lib.pc_last_error(ix._h).decode())
            smp.engine_state = st_c.value
            return cnt_c.value
        # same answers as the buffer API on a planner-sized batch: device samples -> pc_nearest_batch -> host steering -> pc_radius_batch
        chk = PcSampler.make(start, (0.8 * half, 0.5 * half, 2.0), (-half, half, -half, half, 0.0, 4.0), PARAMS["sample_range"], 0.6, 0.3, 0.1, engine_state=4242)
        kc = 200_000
        s_host = ix.sample_batch(chk, kc, advance=False)
        cand = ix.expand_batch(nodes_ix, node_coord, node_radius, node_valid, chk, P, 0.0, 0.6, kc, advance=False)
        with PointCloudIndex(max_points=1 << 16, device=local) as nodes_chk:
            nodes_chk.build(node_coord.astype(np.float32))
            nn, _ = nodes_chk.nearest(s_host.astype(np.float32))
        cn = node_coord[nn]
        d = cn - s_host
        dis = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
        rad = node_radius[nn].astype(np.float64)
        far = dis > rad
        ctr = np.where(far[:, None], cn + (s_host - cn) * (rad / np.where(far, dis, 1.0))[:, None], s_host)
        rr = ix.radius(ctr.astype(np.float32), P)
        keep = ~((ctr[:, 2] < 0.0) | (rr.astype(np.float64) < 0.6))
        dg_same = bool(len(cand) == int(keep.sum()) and (cand["center"] == ctr[keep]).all() and (cand["radius"] == rr[keep]).all())
        for _ in range(2):
            step_expand(M)
        barrier()
        dg_steps = max(3, min(args.steps, 8))
        t0 = time.perf_counter()
        n_cand = 0
        for _ in range(dg_steps):
            n_cand += step_expand(M)
        dg_s = max_over_ranks(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for _ in range(50):
            step_expand(4096)
        small_us = (time.perf_counter() - t0) / 50 * 1e6
        dg = {"value": world * M * dg_steps / dg_s, "unit": "samples/s", "samples_per_call": M, "node_set": n_nodes,
              "candidates_per_call": n_cand // dg_steps, "h2d_bytes_per_call": n_nodes * 29, "d2h_bytes_per_call": 32 * (n_cand // dg_steps) + 12,
              "matches_buffer_api": dg_same, "planner_batch_4096_us": small_us,
              "how": "pc_expand_batch: samples generated on the device from the engine state, nearest vertex + steering + radiusSearch + "
                     "the loop's early rejections on the device; host clock around the call, result in host memory"}

    # strong scaling (N > 1): ONE batch of N x M queries against the time rank 0 needs for the whole batch alone, split two ways:
    #  (a) contiguous slices (pc_shard_range): every rank reads and answers only its N-th of the array -- a random, N times
    #      sparser sample of the batch, so packets are less coherent, but nothing is replicated;
    #  (b) pc_batch_shard: every rank passes over the whole batch and answers the queries whose cell hashes to it -- dense
    #      shares, at the price of a full-batch pass per rank.  (b) wins when a search is expensive (C5: unbounded nearest on
    #      100 M points), (a) for cheap bounded radius queries like this workload; both are reported.
    strong = None
    if world > 1:
        Mt = M * world
        q_all = torch.empty((Mt, 3), dtype=torch.float32, device=dev)
        if rank == 0:
            for r in range(world):
                q_all[r * M:(r + 1) * M].copy_(torch.from_numpy(synth.rrt_queries(M, half, seed=1000 + r)), non_blocking=False)
        dist.broadcast(q_all, 0)
        r_all = torch.full((Mt,), float("nan"), dtype=torch.float32, device=dev)

        from pointcloudtraj_b200 import shard_range
        sb, se = shard_range(Mt, rank, world)

        def step_big(lo=0, hi=Mt):
            rc = lib.pc_radius_batch(ix._h, C.c_void_p(q_all.data_ptr() + 12 * lo), hi - lo, 3, PC_DEVICE, 0, C.byref(P),
                                     C.c_void_p(r_all.data_ptr() + 4 * lo), None)
            if rc != 0:
                raise RuntimeError(lib.pc_last_error(ix._h).decode())

        def timed(n_rep, active, lo=0, hi=Mt):
            for _ in range(2):
                if active:
                    step_big(lo, hi)
            barrier()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            for _ in range(n_rep):
                if active:
                    step_big(lo, hi)
            b_.record()
            torch.cuda.synchronize()
            return max_over_ranks(a_.elapsed_time(b_) * 1e-3) / n_rep

        t1 = timed(5, rank == 0)                       # rank 0 alone, the others idle
        ref_all = r_all.clone()
        dist.broadcast(ref_all, 0)
        r_all.fill_(float("nan"))
        ts = timed(5, True, sb, se)                    # (a) contiguous slices
        slices_ok = torch.tensor([int(bool((r_all[sb:se] == ref_all[sb:se]).all().item()))], device=dev)
        dist.all_reduce(slices_ok, op=dist.ReduceOp.MIN)
        ix.batch_shard(rank, world)
        r_all.fill_(float("nan"))
        tn = timed(5, True)                            # (b) pc_batch_shard
        ix.batch_shard(0, 1)
        # every query answered by exactly one rank (early-outs by all), and with rank 0's value
        mine = ~torch.isnan(r_all)
        cover = mine.to(torch.int32)
        dist.all_reduce(cover)
        okv = torch.tensor([int(bool((r_all[mine] == ref_all[mine]).all().item()))], device=dev)
        dist.all_reduce(okv, op=dist.ReduceOp.MIN)
        best = min(ts, tn)
        strong = {"total_queries": Mt, "one_gpu_ms": t1 * 1e3, "n_gpu_ms": best * 1e3, "value": Mt / best, "unit": UNIT,
                  "efficiency_vs_one_gpu": t1 / (world * best),
                  "split": "contiguous slices (pc_shard_range)" if ts <= tn else "pc_batch_shard (hashed cells), same batch on every rank",
                  "contiguous_slices": {"n_gpu_ms": ts * 1e3, "efficiency_vs_one_gpu": t1 / (world * ts), "matches_one_gpu": bool(slices_ok.item())},
                  "batch_shard": {"n_gpu_ms": tn * 1e3, "efficiency_vs_one_gpu": t1 / (world * tn),
                                  "every_query_answered": bool((cover >= 1).all().item()), "matches_one_gpu": bool(okv.item())}}
        del q_all, r_all, ref_all

    # C3: index rebuild of a 300k-point frame (ms/frame), device-resident frame (rank 0 holds the cloud)
    fms = [0.0] * 12
    if rank == 0:
        frame = t_pts[:FRAME_POINTS].contiguous()
        ixf = PointCloudIndex(max_points=FRAME_POINTS, device=local, stream=stream)
        fms = []
        for _ in range(12):
            ixf.build(frame)
            fms.append(ixf.last_build_ms())
        ixf.close()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        k_ms = float(np.mean(search_ms))
        achieved = BYTES_PER_QUERY * M / (k_ms * 1e-3) / 1e9
        ncu, ncu_note = ncu_figures(M)
        sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        issue_capacity = sm_count * 4 * sm_mhz * 1e6 * k_ms * 1e-3          # warp instructions the 4 schedulers per SM can issue
        roofline_issue = None
        if ncu and ncu.get("inst_executed"):
            roofline_issue = {"bound": "issue", "achieved": ncu["inst_executed"], "peak": issue_capacity, "unit": "warp instructions per launch",
                              "frac": ncu["inst_executed"] / issue_capacity, "source": ncu_note,
                              "how": "smsp__inst_executed.sum of one launch (ncu) / (SMs x 4 schedulers x SM clock x live kernel time)"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": workload_config(args),
                "workload_stats": {"sensing_range_early_out_fraction": early_frac,
                                   "note": "the map (+-36.6 m) is larger than the 31.5 m sensing range around start, so this share of the "
                                           "uniform samples takes radiusSearch's early-out (corridor_finder.cpp:115-116), as in the reference"},
                "device_mode": "PC_DEVICE_ASYNC: steps rotate over 3 internal streams (ordering pass of step k+1 overlaps the search of step k)",
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": (ncu or {}).get("dram_bytes"), "traffic_source": ncu_note,
                             "kernel": "pc_query_packet_kernel<RADIUS, 2> (64-query warp packets over the prefix-split tree)", "kernel_ms": k_ms,
                             "batch_order_ms": float(np.mean(order_ms)),
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                             "algorithmic_bytes_per_query": BYTES_PER_QUERY,
                             "limiter": "not HBM: the index is L2-resident and the kernel is instruction-issue bound -- see roofline_issue"},
                "roofline_issue": roofline_issue,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": 12 * M, "d2h_bytes_per_step": 4 * M,
                        "steps": e2e_steps, "matches_device_result": same,
                        "mode": "PC_HOST_ASYNC, 3 batches in flight, one wait at the end", "blocking_call_value": e2e_blocking,
                        "host_roof_gbs": host_roof_gbs, "host_roof_queries_per_s": host_roof_gbs * 1e9 / 16,
                        "frac_of_host_roof": e2e_val / (host_roof_gbs * 1e9 / 16),
                        "host_roof_how": "all ranks copy one step's 12 B/query in and 4 B/query out from / to pinned memory at once, no kernels"},
                "gpu_launches": launches, "clocks": clocks,
                "index_build_ms_per_frame": {"points": FRAME_POINTS, "median": float(np.median(fms[2:])), "min": float(min(fms))},
                "all_queries_searched": {"value": all_searched_qps, "unit": UNIT, "note": "per GPU, same batch with sample_range = -1 (no early-outs), one stream"},
                "index_build_ms_1M": float(np.median(build_ms[1:])), "index_broadcast_ms": bcast_ms,
                "host_cpu_binding": (f"{len(numa_cpus)} CPUs next to the GPU (NVML affinity)" if numa_cpus else None),
                "replicas_match_root": replica_ok, "strong": strong, "device_generated": dg}
        if not args.no_cpu_baseline and world == 1:
            cb, r_cpu = cpu_baseline(pts, q_host, start, args.cpu_sample)
            cb["gpu_matches_cpu_sample"] = bool((r_cpu.astype(np.float32) == t_r[: len(r_cpu)].cpu().numpy()).all())
            line["cpu_baseline"] = cb
        if r_last is not None:
            dump_outputs(args.dump_outputs, r_last)
        emit(line)
    ix.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_RESULT_FD = None


def emit(line):
    """Write the ONE JSON result line to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


if __name__ == "__main__":
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner at communicator
    # creation, for one) is sent to stderr instead
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
