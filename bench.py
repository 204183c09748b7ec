#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its named config, on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|...] [--dump-outputs DIR]

metric    decoded points/s (whole job, all N GPUs); output GB/s is reported beside it
workload  N=1: BASELINE.json configs[1] -- 10,000 synthetic point clouds x 100,000 points, 14-bit quantized
          positions, delta prediction + wrap, rANS symbols (scheme chosen by the upstream selection rule);
          N>1: the same batch PER GPU (work shards by buffer, no collective: weak scaling)
step      one pass of the attribute-decode hot path over the whole batch
value     inputs (compressed bytes + stream descriptors) resident in HBM when the timed region starts
e2e       the same metric through the public call with HOST buffers: index + H2D + kernels + D2H per step
          (the device listed 8 times in dcb_create = 8 pipeline slices; --e2e-slices)
other     --workload c1 (configs[0], the real asset) | c2tagged | c3 | c4 | c4tagged (configs[1] Tagged, [2], [3]);
          --sweep (configs[4])
roofline  algorithmic bytes (compressed in + decoded out, SURVEY.md 8d) of the dominant kernel / its CUDA-event
          duration measured inside the timed steps, against MEASURED_PEAKS.json
cpu_baseline  the CPU oracle (a linear-time port of the reference's algorithm; the C# itself cannot run: no .NET
          in the image, and it cannot decode point clouds at all) on a bounded sample, all host cores

--impl reference times that CPU oracle as the reference arm (the one other place oracle/ is executed).
--dump-outputs DIR  after the timed steps, what the last step decoded (see sample_outputs), so that two builds can be
          compared output for output: the inputs are generated from fixed seeds.

bench.py runs against the libraries build() left in the tree and writes nothing there.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (clouds per GPU, points per cloud, generator kwargs, description)
    "c2": (10000, 100000, dict(pos_bits=14, scheme=-1),
           "BASELINE configs[1]: 10k point clouds x 100k points, 14-bit positions, delta+wrap, rANS (upstream scheme rule)"),
    "c2raw": (10000, 100000, dict(pos_bits=14, scheme=1), "configs[1] with the Raw scheme forced"),
    "c2tagged": (10000, 100000, dict(pos_bits=14, scheme=0), "configs[1] with the Tagged scheme forced"),
    "c3": (10000, 100000, dict(pos_bits=14, scheme=-1, normal_bits=10, colors=1),
           "BASELINE configs[2]: configs[1] + 10-bit octahedral normals + 8-bit RGB"),
    "c2s": (7000, 100000, dict(pos_bits=14, scheme=-1), "configs[1] shape with 7,000 clouds (experiment)"),
    "small": (1024, 100000, dict(pos_bits=14, scheme=-1), "CI-sized configs[1]: 1,024 clouds x 100k points"),
    "tiny": (64, 20000, dict(pos_bits=14, scheme=-1), "smoke-sized"),
}
# BASELINE configs[3]: meshes per GPU, grid side (side^2 vertices each), description
MESH_WORKLOADS = {
    "c4": (64, 1000, "BASELINE configs[3]: Edgebreaker meshes of 1,000 x 1,000 vertices (1,996,002 faces), connectivity maps "
                     "from the host, 14-bit positions, parallelogram + wrap, rANS (upstream scheme rule)", -1),
    "c4tagged": (64, 1000, "configs[3] with the Tagged scheme forced", 0),
    "c4s": (8, 300, "configs[3] at CI size: 8 meshes of 300 x 300 vertices", -1),
    # SURVEY 8f-3 predictors at configs[3] size: what upstream encoders write at their slowest speeds
    "c4cmp": (64, 1000, "configs[3] shape with the 8f-3 predictors: positions by ConstrainedMultiParallelogram + wrap, normals by "
                        "GeometricNormal + canonicalized octahedron transform (10 bits), Raw rANS; ONE 1,000 x 1,000 mesh written by "
                        "the test suite's bitstream writer (tests/drc_writer.py), repeated 64 times", 1),
    "c4cmps": (8, 300, "c4cmp at CI size: 8 meshes of 300 x 300 vertices", 1),
}
METRIC = "decoded points/sec"
UNIT = "points/s"


def host_buffer(nbytes):
    """Pinned host memory for the e2e leg; pageable (and said so in the JSON line) if the host refuses to pin it."""
    import torch
    try:
        return torch.empty(nbytes, dtype=torch.uint8, pin_memory=True), True
    except RuntimeError:
        return torch.empty(nbytes, dtype=torch.uint8), False


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def make_workload(name, rank, unique, arena_out=None):
    """Synthetic batch for one rank.  `unique` distinct clouds are generated (seed 0xD5AC0000 + rank*2^20 + k) and
    tiled to the batch size with neighbours always distinct (copy j of cloud u sits at index j*unique + u)."""
    from draco_sharp_b200 import synth_gen as G
    n_bufs, n_points, kw, _ = WORKLOADS[name]
    u = n_bufs if unique <= 0 else min(unique, n_bufs)
    spec = G.make_spec(n_points, seed=rank_seed(rank), **kw)
    arena_u, offs_u, lens_u, sums_u, schemes_u, used_u = G.synth_batch(spec, u, n_threads=host_cores())
    if u == n_bufs:
        return arena_u, offs_u, lens_u, sums_u, schemes_u, used_u
    reps = (n_bufs + u - 1) // u
    stride = (used_u + 15) // 16 * 16
    total = stride * reps
    arena = arena_out(total) if arena_out else np.empty(total, dtype=np.uint8)
    offs = np.zeros(n_bufs, dtype=np.uint64)
    lens = np.zeros(n_bufs, dtype=np.uint64)
    sums = np.zeros((n_bufs, 3), dtype=np.uint64)
    schemes = np.zeros((n_bufs, 3), dtype=np.int32)
    for j in range(reps):
        arena[j * stride: j * stride + used_u] = arena_u[:used_u]
        lo = j * u
        hi = min(n_bufs, lo + u)
        offs[lo:hi] = offs_u[: hi - lo] + np.uint64(j * stride)
        lens[lo:hi] = lens_u[: hi - lo]
        sums[lo:hi] = sums_u[: hi - lo]
        schemes[lo:hi] = schemes_u[: hi - lo]
    return arena, offs, lens, sums, schemes, total


def reduce_over_ranks(dist, device, ms, sums):
    """Multi-GPU bookkeeping: the step time is the MAX over ranks, the work counters are SUMMED (whole-job value).
    `dist` is torch.distributed (or None for one process); `sums` is a list of per-rank counters."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return ms, list(sums)
    import torch
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    v = torch.tensor([float(x) for x in sums], dtype=torch.float64, device=device)
    dist.all_reduce(v, op=dist.ReduceOp.SUM)
    return float(t.item()), [float(x) for x in v.tolist()]


def rank_seed(rank):
    """Every rank decodes its own, distinct batch (work shards by buffer: weak scaling, no collective on the data path).
    DCB_BENCH_DATA_RANK=r: a one-GPU run decodes the batch rank r of a multi-GPU run would get."""
    rank = int(os.environ.get("DCB_BENCH_DATA_RANK", rank))
    return 0xD5AC0000 + (rank << 20)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []
        self.first = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Samples from here on belong to the timed region."""
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw = [], [], []
        reasons = set()
        lines = self.lines[self.first:] if len(self.lines) - self.first >= 2 else self.lines[-3:]
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(workload)
        except Exception:
            return None
    return None


DUMP_BUDGET = 60 << 20  # payload bytes of --dump-outputs; with the .npy headers the files stay under 64 MB


def widened(dtype):
    """float32 holds float32 and 8/16-bit integers exactly, float64 holds 32-bit integers exactly."""
    dtype = np.dtype(dtype)
    return np.dtype(np.float32 if dtype == np.float32 or dtype.itemsize <= 2 else np.float64)


def sample_outputs(batch, fetch):
    """The decoded attributes of a fixed, seeded sample of the batch's buffers, as a caller receives them
    (PointAttribute.values: entries x components).  Buffers are taken in a seeded order until DUMP_BUDGET is reached.
    fetch(off, nbytes) returns those bytes of the output arena.  Returns {buffer index: [array per attribute]}."""
    from draco_sharp_b200.decoder import NP_DTYPES
    out, used = {}, 0
    for k in np.random.default_rng(0xD0D0).permutation(batch.n_bufs).tolist():
        infos = [batch.attr_info(k, a) for a in range(batch.buffer_info(k).n_attrs)]
        size = sum(ai.n_entries * ai.num_components * widened(NP_DTYPES[ai.data_type]).itemsize for ai in infos)
        if used + size > DUMP_BUDGET:
            break
        used += size
        out[k] = [fetch(ai.out_off, ai.out_bytes).view(NP_DTYPES[ai.data_type]).reshape(ai.n_entries, ai.num_components)
                  for ai in infos]
    return out


def write_outputs(dirname, outputs):
    """DIR/buf<k>_attr<a>.npy per attribute of sample_outputs(), widened to float32 / float64 without rounding."""
    os.makedirs(dirname, exist_ok=True)
    for k, arrays in outputs.items():
        for a, v in enumerate(arrays):
            np.save(os.path.join(dirname, "buf%05d_attr%d.npy" % (k, a)), v.astype(widened(v.dtype)))


def cpu_oracle_rate(workload, seconds_target=15.0, threads=None):
    """The CPU oracle on a bounded sample of the same workload, one buffer per thread.  Returns points/s etc."""
    from oracle import pyoracle as O  # cpu_baseline / reference arm only
    from draco_sharp_b200 import synth_gen as G
    O.lib()
    n_bufs, n_points, kw, _ = WORKLOADS[workload]
    threads = threads or host_cores()
    # ~1e7 points/s/core for positions only: size the sample for about seconds_target core-seconds
    per_cloud = n_points * (1 + (1 if kw.get("normal_bits") else 0) + (1 if kw.get("colors") else 0))
    n_sample = int(max(threads, min(n_bufs, seconds_target * 0.8e7 / max(per_cloud, 1))))
    n_sample = max(threads, (n_sample // threads) * threads)
    spec = G.make_spec(n_points, seed=0xD5AC0000, **kw)
    arena, offs, lens, _, _, _ = G.synth_batch(spec, n_sample, n_threads=threads)
    chunks = [(offs[t::threads], lens[t::threads]) for t in range(threads)]
    results = [None] * threads

    def work(t):
        results[t] = O.decode_bench(arena, chunks[t][0], chunks[t][1])

    def run():
        th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        return time.perf_counter() - t0

    return n_sample, n_points, threads, run, results


def run_reference(args, rank, world):
    """Reference arm: the reference's own algorithm on the host CPU (oracle port; the C# needs .NET, absent)."""
    if rank != 0:
        return
    if args.workload == "c1":
        from oracle import pyoracle as O
        buf = np.fromfile(os.path.join(ROOT, "tests", "golden", "house_04.obj.drc"), dtype=np.uint8)
        r = O.decode(buf)
        steps = args.steps
        t0 = time.perf_counter()
        for _ in range(steps):
            O.decode(buf)
        ms = (time.perf_counter() - t0) * 1e3 / steps
        n = int(r.n_points)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": n / (ms * 1e-3), "unit": UNIT, "n_gpus": args.gpus,
                          "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "i32->f32", "data": "real asset",
                          "config": {"workload": "c1", "description": "house_04.obj.drc, whole file (3 attributes), 1 buffer"},
                          "cpu_baseline": {"value": n / (ms * 1e-3), "unit": UNIT, "cores": 1, "kind": "port", "sample": "the whole buffer"},
                          "e2e": {"value": n / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    mesh = args.workload in MESH_WORKLOADS
    if mesh:
        n_sample, n_points, threads, run, results = cpu_mesh_rate(args.workload)
    else:
        n_sample, n_points, threads, run, results = cpu_oracle_rate(args.workload, seconds_target=20.0)
    for _ in range(max(1, min(args.warmup, 1))):
        run()
    times = [run() for _ in range(max(1, args.steps))]
    dt = float(np.mean(times))
    pts = sum(r[0] for r in results)
    outb = sum(r[1] for r in results)
    val = pts / dt
    n_bufs = (MESH_WORKLOADS if mesh else WORKLOADS)[args.workload][0]
    desc = MESH_WORKLOADS[args.workload][2] if mesh else WORKLOADS[args.workload][3]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32->f32", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc,
                   "clouds_per_gpu": n_bufs, "points_per_cloud": n_points},
        "output_GBps": outb / dt / 1e9,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d of the workload's clouds x %d points per step, one buffer per thread; C oracle "
                                   "-O2 (linear-time port of the C# algorithm; the C# is O(n^2) and throws on point clouds)" % (n_sample, n_points)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def make_cmp_mesh(side, topo):
    """One grid mesh with CMP positions and geometric normals (SURVEY 8f-3), written by tests/drc_writer.py; cached in the
    temporary directory (the tree may be read-only) because the pure-Python writer needs about a minute per million
    vertices.  Returns (buffer, attr_section_off, checksum of the expected position floats, 1, None)."""
    import struct
    from draco_sharp_b200 import synth_gen as G
    cache = os.path.join(tempfile.gettempdir(), "draco_sharp_b200_bench_%d" % os.getuid(), "c4cmp_%d.npz" % side)
    if os.path.exists(cache):
        z = np.load(cache)
        return z["buf"], int(z["aoff"]), int(z["sum"]), 1, None
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import drc_writer as W
    rng = np.random.default_rng(0xC4C)
    n, bits = side * side, 14
    yy, xx = np.mgrid[0:side, 0:side]
    z = 8000 + 6000 * np.sin(xx / 37.0) * np.cos(yy / 53.0) + rng.normal(0.0, 6.0, size=xx.shape)
    step = ((1 << bits) - 200) // side
    surf = np.stack([xx * step + rng.integers(0, 3, size=xx.shape), yy * step + rng.integers(0, 3, size=xx.shape),
                     z.astype(np.int64)], axis=-1).reshape(-1, 3)
    q = np.zeros_like(surf)
    q[topo["vertex_to_data"]] = surf   # entry order
    q = q.ravel()
    hi = (1 << bits) - 1
    corr, crease = W.cmp_encode(q, 3, topo, 0, hi, rng, 0.15)
    sec = bytearray([1, 0xFF, 0, 0])
    sec += W.varint(2) + bytes([0, 9, 3, 0]) + W.varint(0) + bytes([1, 9, 3, 0]) + W.varint(1) + bytes([2, 3])
    sec += W.portable_int(corr, 3, 4, 1, "raw", W.cmp_data(crease, 0, hi))
    sec += W.portable_int(rng.integers(0, 24, size=n * 2), 2, 6, 3, "raw", W.geometric_normal_data(rng.integers(0, 2, size=n) < 1, 10), zig=False)
    pos_min, rng_f = np.float32(-1.0), np.float32(2.0)
    sec += W.quant_params([-1.0, -1.0, -1.0], 2.0, bits) + bytes([10])
    head = b"DRACO" + bytes([2, 2, 1, 1]) + struct.pack("<H", 0) + bytes([0]) + b"\xEB" * 15  # connectivity: the host's business
    buf = np.frombuffer(head + bytes(sec), dtype=np.uint8).copy()
    delta = np.float32(rng_f / np.float32(hi))
    fl = (q.astype(np.float32) * delta).astype(np.float32) + pos_min   # two separately rounded binary32 operations
    sm = G.word_checksum(fl.astype(np.float32))
    os.makedirs(os.path.dirname(cache), exist_ok=True)
    np.savez(cache, buf=buf, aoff=len(head), sum=np.uint64(sm))
    return buf, len(head), int(sm), 1, None


def make_meshes(name, rank, n_meshes=None):
    from concurrent.futures import ThreadPoolExecutor
    from draco_sharp_b200 import synth_gen as G
    m, side, _, scheme = MESH_WORKLOADS[name]
    m = n_meshes or m
    topo = G.grid_topology(side, side)
    if name.startswith("c4cmp"):
        one = make_cmp_mesh(side, topo)
        return topo, [one] * m, side * side
    with ThreadPoolExecutor(max_workers=host_cores()) as ex:
        meshes = list(ex.map(lambda k: G.grid_mesh(side, side, topo, seed=rank_seed(rank) + 0x4000 + k, scheme=scheme), range(m)))
    return topo, meshes, side * side


def cpu_mesh_rate(name, threads=None):
    """CPU oracle on the mesh workload: one mesh per thread, maps handed over exactly as to the GPU path."""
    from oracle import pyoracle as O  # cpu_baseline / reference arm only
    O.lib()
    threads = threads or host_cores()
    topo, meshes, nv = make_meshes(name, 0, n_meshes=threads)
    results = [None] * threads

    def work(t):
        buf, aoff, sm, _, _ = meshes[t]
        r = O.decode(buf, [topo], aoff, nv)
        assert r.status == 0
        results[t] = (nv, r.attrs[0].out.nbytes)

    def run():
        th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        return time.perf_counter() - t0

    return threads, nv, threads, run, results


def run_mesh(args, rank, local_rank, world):
    """configs[3]: a batch of large meshes.  Connectivity (corner table + traversal maps) comes from the host, the
    symbol decode, parallelogram inverse prediction, wrap and dequantisation run on the GPU."""
    import torch
    import draco_sharp_b200 as D
    from draco_sharp_b200 import synth_gen as G
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the decode path is CUDA only (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    args.warmup = max(args.warmup, 3)
    t0 = time.perf_counter()
    topo, meshes, nv = make_meshes(args.workload, rank, args.meshes or None)
    gen_s = time.perf_counter() - t0
    bufs = [m[0] for m in meshes]
    dec = D.DracoBatchDecoder([local_rank])
    stream = torch.cuda.current_stream()
    dec.set_stream(0, stream.cuda_stream)

    def indexed():
        b = dec.index(bufs)
        for k, m in enumerate(meshes):
            b.set_attr_section(k, m[1], nv)
            b.set_mesh_maps(k, 0, topo["opposite"], topo["corner_to_vertex"], topo["data_to_corner"], topo["vertex_to_data"])
        b.finish()
        return b

    batch = indexed()
    n_bufs, points, out_bytes, in_bytes, algo_bytes = batch.n_bufs, batch.points, batch.out_bytes, batch.in_bytes, batch.algo_bytes
    maps_bytes = sum(int(v.nbytes) for v in topo.values()) * n_bufs
    dec.upload(batch)
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")

    def step():
        dec.decode_resident(batch, dev_out=d_out.data_ptr())

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step()
    for k in range(n_bufs):
        assert batch.status(k) == 0, "mesh %d failed: %d" % (k, batch.status(k))
        ai = batch.attr_info(k, 0)
        got = d_out[ai.out_off: ai.out_off + ai.out_bytes].cpu().numpy()
        assert G.word_checksum(got) == meshes[k][2], "decoded positions of mesh %d do not match the generator" % k
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dom_ms, launches = [], 0
    ev0.record(stream)
    for _ in range(args.steps):
        step()
        st = dec.stats()
        dom_ms.append(st.ms_dominant)
        launches += st.n_launches
    ev1.record(stream)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, sample_outputs(batch, lambda off, n: d_out[off: off + n].cpu().numpy()))
    ms, (total_points, total_out, total_launches) = reduce_over_ranks(dist, "cuda", ev0.elapsed_time(ev1), [points, out_bytes, launches])
    ms_per_step = ms / args.steps
    stats = dec.stats()
    # e2e: index + maps + H2D (buffers and maps) + kernels + D2H
    h_out, _ = host_buffer(out_bytes)
    e2e_ms = []
    for i in range(args.e2e_steps + 1):
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        b2 = indexed()
        dec.decode(b2, out_ptr=h_out.data_ptr())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        b2.free()
        if i > 0:
            e2e_ms.append(dt)
    e2e_t = float(np.mean(e2e_ms)) if e2e_ms else float("nan")
    e2e_t, _ = reduce_over_ranks(dist, "cuda", e2e_t, [0.0])
    if e2e_ms:
        ai = batch.attr_info(n_bufs // 2, 0)
        assert G.word_checksum(h_out.numpy()[ai.out_off: ai.out_off + ai.out_bytes]) == meshes[n_bufs // 2][2]
    if rank == 0:
        peak, peak_src = measured_peak()
        dom = float(np.mean(dom_ms)) if dom_ms else 0.0
        dom_bytes = int(stats.algo_bytes_dominant) or algo_bytes
        achieved = (dom_bytes / (dom * 1e-3) / 1e9) if dom > 0 else 0.0
        line = {
            "metric": METRIC, "value": total_points / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32->f32", "data": "synthetic",
            "config": {"workload": args.workload, "description": MESH_WORKLOADS[args.workload][2], "meshes_per_gpu": n_bufs,
                       "vertices_per_mesh": nv, "faces_per_mesh": int(topo["opposite"].size // 3),
                       "symbol_scheme_of_positions": {0: "tagged", 1: "raw"}.get(meshes[0][3], "n/a"),
                       "compressed_bytes_per_gpu": in_bytes, "output_bytes_per_gpu": out_bytes, "map_bytes_per_gpu": maps_bytes,
                       "l2": "inputs+outputs+maps (%.1f GB per step) exceed the 126 MB L2" % ((in_bytes + out_bytes + maps_bytes) / 1e9),
                       "generate_s": round(gen_s, 1)},
            "output_GBps": total_out / (ms_per_step * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                         "traffic": profile_traffic(args.workload), "peak_source": peak_src,
                         "kernel": stats.dominant_name.decode(), "kernel_ms": dom, "algorithmic_bytes_per_launch": dom_bytes,
                         "algorithmic_bytes_per_step": algo_bytes,
                         "stage_ms": {"raw_fused": stats.ms_raw, "tag_rans": stats.ms_tag, "par_post": stats.ms_par,
                                      "parallelogram": stats.ms_para, "all_kernels": stats.ms_total},
                         "stage_ms_what": "parallelogram = the whole mesh-prediction stage behind the rANS kernels (parallelogram / "
                                          "constrained multi-parallelogram / tex-coord / geometric-normal kernels), one timed span",
                         "note": "one serial rANS chain of %d symbols and one serial prediction chain per mesh attribute "
                                 "(dependency depth of a depth-first traversal ~ 0.86 n): %d meshes in flight" % (3 * nv, n_bufs)},
            "e2e": {"value": total_points / (e2e_t * 1e-3), "unit": UNIT, "h2d_bytes_per_step": in_bytes + maps_bytes,
                    "d2h_bytes_per_step": out_bytes, "ms_per_step": e2e_t, "steps": args.e2e_steps,
                    "what": "dcb_index + dcb_set_mesh_maps + dcb_index_finish + dcb_decode: host indexing, H2D of buffers and maps, kernels, D2H"},
            "gpu_launches": int(total_launches), "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            n_sample, n_points, threads, run, results = cpu_mesh_rate(args.workload)
            run()
            dt = run()
            line["cpu_baseline"] = {"value": sum(r[0] for r in results) / dt, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "%d meshes x %d vertices of the same workload, one mesh per thread, C oracle -O2" % (n_sample, n_points)}
        print(json.dumps(line), flush=True)
    batch.free()
    dec.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def run_real_asset(args, rank, local_rank):
    """BASELINE configs[0]: the reference's one real asset (house_04.obj.drc: Edgebreaker mesh, 11-bit positions,
    parallelogram + wrap, Raw rANS; texture coordinates with the TexCoordsPortable predictor; a generic uint8 attribute),
    bytes verbatim.  Whole decode through the public call: host Edgebreaker connectivity (CPU by design), indexing,
    H2D, kernels, D2H.  3,220 points: latency, not throughput."""
    if rank != 0:
        return
    import torch
    import draco_sharp_b200 as D
    from oracle import pyoracle as O  # cpu_baseline only
    buf = np.fromfile(os.path.join(ROOT, "tests", "golden", "house_04.obj.drc"), dtype=np.uint8)
    torch.cuda.set_device(local_rank)
    dec = D.DracoBatchDecoder([local_rank])
    ref = O.decode(buf)
    assert ref.status == 0
    for _ in range(max(3, args.warmup)):
        (d,) = dec.decode_batch([buf])
    assert d.ok and len(d.attributes) == 3, "GPU decode failed"
    for k in range(3):
        assert np.array_equal(np.asarray(d.attributes[k].buffer).view(np.uint8).ravel(), ref.attrs[k].out.view(np.uint8).ravel()), \
            "GPU decode differs from the oracle (attribute %d)" % k
    steps = args.steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        (d,) = dec.decode_batch([buf])
    ms = (time.perf_counter() - t0) * 1e3 / steps
    st = dec.stats()
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {0: [a.values for a in d.attributes]})
    t0 = time.perf_counter()
    for _ in range(steps):
        O.decode(buf)
    cpu_ms = (time.perf_counter() - t0) * 1e3 / steps
    n = int(ref.n_points)
    out_bytes = int(sum(ref.attrs[k].out.nbytes for k in range(3)))
    print(json.dumps({
        "metric": METRIC, "value": n / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32->f32", "data": "real asset",
        "config": {"workload": "c1", "description": "BASELINE configs[0]: house_04.obj.drc (reference sample), whole file verbatim: positions, "
                   "tex coords, generic uint8; 1 buffer, %d points, %d faces" % (n, len(d.faces))},
        "e2e": {"value": n / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(buf.nbytes), "d2h_bytes_per_step": out_bytes,
                "ms_per_step": ms, "what": "dcb_index + dcb_host_connectivity + dcb_index_finish + dcb_decode"},
        "roofline": {"bound": "hbm", "achieved": None, "peak": measured_peak()[0], "unit": "GB/s", "frac": None, "traffic": None,
                     "note": "three small streams of one mesh: launch latency and host work, kernels %.3f ms of %.3f ms" % (st.ms_total, ms)},
        "cpu_baseline": {"value": n / (cpu_ms * 1e-3), "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "the same buffer, C oracle -O2 (connectivity + attribute), %.3f ms per decode" % cpu_ms},
        "gpu_launches": int(st.n_launches) * steps}), flush=True)
    dec.close()


def run_sweep(args, rank, local_rank):
    """BASELINE configs[4]: points-per-buffer sweep (total points fixed) and batch-size sweep (points per buffer fixed).
    Kernel-only numbers (inputs resident), one JSON line per cell; not the headline."""
    import torch
    import draco_sharp_b200 as D
    from draco_sharp_b200 import synth_gen as G
    torch.cuda.set_device(local_rank)
    dec = D.DracoBatchDecoder([local_rank])
    stream = torch.cuda.current_stream()
    dec.set_stream(0, stream.cuda_stream)
    peak, _ = measured_peak()
    cells = [("points_per_buffer", n, max(1, 200_000_000 // n)) for n in (1000, 10_000, 100_000, 1_000_000, 10_000_000)]
    cells += [("batch_size", 100_000, b) for b in (1, 16, 256, 4096, 16384, 65536)]
    for scheme, sname in ((1, "raw"), (0, "tagged")):
        for axis, n, b in cells:
            uniq = min(b, max(1, 20_000_000 // n))
            spec = G.make_spec(n, seed=rank_seed(rank) + n, pos_bits=14, scheme=scheme)
            arena_u, offs_u, lens_u, sums_u, schemes_u, used_u = G.synth_batch(spec, uniq, n_threads=host_cores())
            reps = (b + uniq - 1) // uniq
            stride = (used_u + 15) // 16 * 16
            arena = np.empty(stride * reps, dtype=np.uint8)
            offs = np.zeros(b, dtype=np.uint64)
            lens = np.zeros(b, dtype=np.uint64)
            for j in range(reps):
                arena[j * stride: j * stride + used_u] = arena_u[:used_u]
                lo, hi = j * uniq, min(b, (j + 1) * uniq)
                offs[lo:hi] = offs_u[: hi - lo] + np.uint64(j * stride)
                lens[lo:hi] = lens_u[: hi - lo]
            batch = dec.index_arena(arena, offs, lens)
            dec.upload(batch)
            d_out = torch.empty(batch.out_bytes, dtype=torch.uint8, device="cuda")
            for _ in range(3):
                dec.decode_resident(batch, dev_out=d_out.data_ptr())
            ai = batch.attr_info(0, 0)
            ok = G.word_checksum(d_out[ai.out_off: ai.out_off + ai.out_bytes].cpu().numpy()) == int(sums_u[0, 0])
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            steps = 5
            torch.cuda.synchronize()
            ev0.record(stream)
            for _ in range(steps):
                dec.decode_resident(batch, dev_out=d_out.data_ptr())
            ev1.record(stream)
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / steps
            st = dec.stats()
            # one write per line: under torchrun the ranks share a stdout
            sys.stdout.write(json.dumps({"sweep": axis, "scheme": sname, "rank": rank, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
                              "points_per_buffer": n, "buffers": b, "ms_per_step": ms,
                              "points_per_s": batch.points / (ms * 1e-3), "algorithmic_GBps": batch.algo_bytes / (ms * 1e-3) / 1e9,
                              "frac_of_hbm_peak": batch.algo_bytes / (ms * 1e-3) / 1e9 / peak, "parity_ok": bool(ok),
                              "launches": st.n_launches, "stage_ms": {"raw": st.ms_raw, "tag": st.ms_tag, "par": st.ms_par}}) + "\n")
            sys.stdout.flush()
            batch.free()
            del d_out
    dec.close()


def positive(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=60, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + sorted(MESH_WORKLOADS) + ["c1"])
    ap.add_argument("--unique", type=int, default=2048, help="distinct clouds generated per rank (0 = all distinct)")
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--e2e-slices", type=int, default=8, help="pipeline slices of the e2e leg (dcb_create with the device listed K times)")
    ap.add_argument("--meshes", type=int, default=0, help="mesh workloads: meshes per GPU (0 = the workload's default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-copy-ceiling", action="store_true", help="skip the bare pinned-copy leg (e2e.host_ceiling_*)")
    ap.add_argument("--sweep", action="store_true", help="BASELINE configs[4]: points-per-buffer and batch-size sweep (one JSON line per cell)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the decoded attributes of the last step "
                    "(a fixed sample of the buffers, at most 64 MB; rank 0's batch) as DIR/buf<k>_attr<a>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.sweep):
        ap.error("--dump-outputs needs the GPU arm of a workload (not --impl reference, not --sweep)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.sweep:
        return run_sweep(args, rank, local_rank)
    if args.workload == "c1":
        return run_real_asset(args, rank, local_rank)
    if args.workload in MESH_WORKLOADS:
        return run_mesh(args, rank, local_rank, world)
    args.warmup = max(args.warmup, 3)

    import torch
    import draco_sharp_b200 as D
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the decode path is CUDA only (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()

    # ---- synthetic inputs, host side (pinned, so the e2e leg copies at full PCIe speed) ----
    t0 = time.perf_counter()
    pinned = {}

    def pinned_arena(nbytes):
        pinned["in"], pinned["in_ok"] = host_buffer(nbytes)
        return pinned["in"].numpy()

    arena, offs, lens, sums, schemes, used = make_workload(args.workload, rank, args.unique, pinned_arena)
    if "in" not in pinned:  # all-distinct path returned a pageable arena
        pinned["in"], pinned["in_ok"] = host_buffer(used)
        pinned["in"].numpy()[:] = arena[:used]
        arena = pinned["in"].numpy()
    gen_s = time.perf_counter() - t0

    dec = D.DracoBatchDecoder([local_rank])
    stream = torch.cuda.current_stream()
    dec.set_stream(0, stream.cuda_stream)
    batch = dec.index_arena(arena, offs, lens)
    n_bufs = batch.n_bufs
    points = batch.points
    out_bytes = batch.out_bytes
    in_bytes = batch.in_bytes
    algo_bytes = batch.algo_bytes
    dec.upload(batch)
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")

    def step():
        dec.decode_resident(batch, dev_out=d_out.data_ptr())

    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi needs ~0.5 s to come up: start it before the warm-up, keep the samples under load
    for _ in range(args.warmup):
        step()
    # parity gate before any number is reported: word checksums of a sample of decoded attributes
    from draco_sharp_b200 import synth_gen as G
    nocheck = bool(os.environ.get("DCB_BENCH_NOCHECK"))  # kernel experiments only
    for k in ([] if nocheck else list(range(0, n_bufs, max(1, n_bufs // 16)))[:16]):
        assert batch.status(k) == 0, "buffer %d failed: %d" % (k, batch.status(k))
        ai = batch.attr_info(k, 0)
        got = d_out[ai.out_off: ai.out_off + ai.out_bytes].cpu().numpy()
        assert G.word_checksum(got) == int(sums[k, 0]), "decoded positions of buffer %d do not match the generator" % k
    bad = sum(1 for k in range(n_bufs) if batch.status(k) != 0)
    assert bad == 0, "%d buffers failed" % bad

    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    sampler.mark()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    dom_ms = []
    launches = 0
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
        st = dec.stats()
        dom_ms.append(st.ms_dominant)
        launches += st.n_launches
    ev1.record(stream)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, sample_outputs(batch, lambda off, n: d_out[off: off + n].cpu().numpy()))
    ms, (total_points, total_out, total_launches) = reduce_over_ranks(dist, "cuda", ev0.elapsed_time(ev1),
                                                                      [points, out_bytes, launches])
    total_launches = int(total_launches)
    ms_per_step = ms / args.steps
    value = total_points / (ms_per_step * 1e-3)
    stats = dec.stats()

    # ---- e2e: host buffers in, host buffers out, through the public call (index + H2D + kernels + D2H) ----
    # the same device listed K times = K pipeline slices: H2D, kernels and D2H of neighbouring slices overlap
    h_out, out_pinned = host_buffer(out_bytes)
    dec_e2e = D.DracoBatchDecoder([local_rank] * max(1, args.e2e_slices)) if args.e2e_slices > 1 else dec
    e2e_ms = []
    for i in range(args.e2e_steps + 1):
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        b2 = dec_e2e.index_arena(arena, offs, lens)
        dec_e2e.decode(b2, out_ptr=h_out.data_ptr())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        if i == 0:
            e2e_offs = [(b2.attr_info(k, 0).out_off, b2.attr_info(k, 0).out_bytes) for k in (0, n_bufs // 2, n_bufs - 1)]
        b2.free()
        if i > 0:
            e2e_ms.append(dt)
    e2e_t = float(np.mean(e2e_ms)) if e2e_ms else float("nan")
    e2e_t, _ = reduce_over_ranks(dist, "cuda", e2e_t, [0.0])
    for k, (oo, ob) in zip((0, n_bufs // 2, n_bufs - 1), e2e_offs):
        assert nocheck or G.word_checksum(h_out.numpy()[oo: oo + ob]) == int(sums[k, 0]), "e2e output of buffer %d is wrong" % k
    if dec_e2e is not dec:
        dec_e2e.close()
    e2e_value = total_points / (e2e_t * 1e-3)

    # ---- what the host side of this box can do at all: the e2e leg's bytes as BARE pinned copies, all ranks at once
    # (H2D and D2H on a stream each, overlapping as in the decode pipeline; no kernels, no indexing).  e2e time over
    # this time says how much of the leg is the link / the host's memory system and how much is ours.
    ceil_ms = float("nan")
    if args.e2e_steps > 0 and not args.no_copy_ceiling:
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        d_in = torch.empty(in_bytes, dtype=torch.uint8, device="cuda")
        h_in_t = pinned["in"][:in_bytes] if len(pinned["in"]) >= in_bytes else None
        ts = []
        for i in range(3):
            torch.cuda.synchronize()
            if dist:
                dist.barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_in):
                if h_in_t is not None:
                    d_in.copy_(h_in_t, non_blocking=True)
            with torch.cuda.stream(s_out):
                h_out.copy_(d_out, non_blocking=True)
            torch.cuda.synchronize()
            if i > 0:
                ts.append((time.perf_counter() - t0) * 1e3)
        del d_in
        ceil_ms, _ = reduce_over_ranks(dist, "cuda", float(np.mean(ts)), [0.0])

    if rank == 0:
        peak, peak_src = measured_peak()
        dom = float(np.mean(dom_ms)) if dom_ms else 0.0
        dom_bytes = int(stats.algo_bytes_dominant) or algo_bytes
        achieved = (dom_bytes / (dom * 1e-3) / 1e9) if dom > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32->f32", "data": "synthetic",
            "config": {"workload": args.workload, "description": WORKLOADS[args.workload][3],
                       "clouds_per_gpu": n_bufs, "points_per_cloud": WORKLOADS[args.workload][1],
                       "unique_clouds_per_gpu": int(n_bufs if args.unique <= 0 else min(args.unique, n_bufs)),
                       "symbol_scheme_of_positions": {0: "tagged", 1: "raw"}.get(int(schemes[0, 0]), "n/a"),
                       "compressed_bytes_per_gpu": in_bytes, "output_bytes_per_gpu": out_bytes,
                       "l2": "inputs+outputs (%.1f GB per step) exceed the 126 MB L2" % ((in_bytes + out_bytes) / 1e9),
                       "generate_s": round(gen_s, 1)},
            "output_GBps": total_out / (ms_per_step * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": profile_traffic(args.workload),
                         "frac_of_8TBps": achieved / 8000.0,
                         "whole_step": {"achieved": algo_bytes / (ms_per_step * 1e-3) / 1e9, "frac": algo_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                                        "what": "algorithmic bytes of the whole step / step time: the figure to compare across workloads "
                                                "(the dominant kernel may share the SMs with the step's other kernels)"},
                         "chain_bound": {"symbols_per_stream": WORKLOADS[args.workload][1] * 3,
                                         "cycles_per_symbol": (dom * 1e-3 * clocks.get("sm_mhz", 0) * 1e6 / (WORKLOADS[args.workload][1] * 3))
                                         if dom > 0 and clocks.get("sm_mhz") else None,
                                         "what": "serial-chain bound of BASELINE.md 3.4: symbols_per_stream x cycles/symbol / clock = kernel_ms "
                                                 "while every stream is resident; more streams per launch do not lengthen it"},
                         "peak_source": peak_src, "kernel": stats.dominant_name.decode(), "kernel_ms": dom,
                         "algorithmic_bytes_per_launch": dom_bytes, "algorithmic_bytes_per_step": algo_bytes,
                         "stage_ms": {"raw_fused": stats.ms_raw, "tag_rans": stats.ms_tag, "par_post": stats.ms_par,
                                      "all_kernels": stats.ms_total},
                         "note": "serial rANS chains: %d streams x %d symbols; residency waves %d, %d lanes/warp, %d B smem/stream"
                                 % (n_bufs, WORKLOADS[args.workload][1] * 3, stats.n_waves, stats.lanes_per_warp, stats.smem_per_stream)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
                    "ms_per_step": e2e_t, "steps": args.e2e_steps, "pipeline_slices": args.e2e_slices,
                    "ms_each": [round(x, 1) for x in e2e_ms],
                    "host_buffers_pinned": bool(out_pinned and pinned.get("in_ok", False)),
                    "host_ceiling_ms": ceil_ms,
                    "host_ceiling_GBps": (world * (in_bytes + out_bytes) / (ceil_ms * 1e-3) / 1e9) if ceil_ms == ceil_ms else None,
                    "frac_of_host_ceiling": (ceil_ms / e2e_t) if ceil_ms == ceil_ms and e2e_t == e2e_t else None,
                    "host_ceiling_what": "the same bytes as bare pinned cudaMemcpyAsync (H2D and D2H on a stream each), all ranks at "
                                         "once: the link and the host memory system alone, max over ranks",
                    "what": "dcb_index_arena + dcb_decode: host indexing, H2D from pinned memory, kernels, D2H to pinned memory"},
            "reference_csharp": "not runnable: no .NET SDK in image (BASELINE.md 3.1); the reference arm is the C oracle port",
            "gpu_launches": total_launches,
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            n_sample, n_points, threads, run, results = cpu_oracle_rate(args.workload)
            run()
            dt = run()
            line["cpu_baseline"] = {
                "value": sum(r[0] for r in results) / dt, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": "%d clouds x %d points of the same workload, one buffer per thread, C oracle -O2" % (n_sample, n_points)}
        print(json.dumps(line), flush=True)
    batch.free()
    dec.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
