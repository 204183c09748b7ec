"""Point order (DCB_ORDER_POINTS) against entry order on the same inputs, one process, on a B200.

Workloads:
  c4        64 Edgebreaker grid meshes of 1,000 x 1,000 vertices (bench.py --workload c4), faces omitted (the NULL form:
            point ids = corner_to_vertex) and explicit faces (= corner_to_vertex, uploaded with the maps)
  house     ~20,000 copies of tests/golden/house_04.obj.drc (~64M points, attribute seams): connectivity decoded once
            by the host helper, installed on every copy with dcb_set_mesh_maps + dcb_set_mesh_faces
Per workload and order, two batches are indexed and uploaded once, then decoded resident in alternation (CUDA events
around each step, after warm-up); e2e is index + connectivity + H2D + kernels + D2H into host memory.  The point
stage's own time comes from a separate torch.profiler run (kernels point_win / point_resolve / point_gather).  A seeded
sample of point-order attributes is checked against a NumPy gather of the entry-order output of the same run.
Writes JSON lines to stdout and to --out (default profiles/point_order_b200.jsonl)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = "unknown"
    return name, q


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6650.0, "bench.py fallback (no MEASURED_PEAKS.json in the tree)"


def build(dec, kind, points, res):
    """Index one batch of the workload in the given order (connectivity installed, index finished)."""
    bufs, conn = res["bufs"], res["conn"]
    b = dec.index(bufs)
    if points:
        b.set_output_order(True)
    for k in range(len(bufs)):
        off, n_points, maps, faces = conn
        b.set_attr_section(k, off, n_points)
        for d, m in enumerate(maps):
            b.set_mesh_maps(k, d, m["opposite"], m["corner_to_vertex"], m["data_to_corner"], m["vertex_to_data"])
        if points:
            b.set_mesh_faces(k, faces)
    b.finish()
    return b


def algo_bytes(res, points_rows):
    """Algorithmic bytes of the point stage from the shapes: corner pass 12 B per corner (point id, vertex id, one
    red.max), zeroing 4 B + resolve 16 B per point and decoder, gather per row 4 B of map + a read and a write of the row."""
    _, n_points, _, _ = res["conn"]
    n = len(res["bufs"])
    corners = sum(int(m["corner_to_vertex"].size) for m in res["used_maps"])
    pts = n_points * len(res["used_maps"])
    gather = sum(rows * (4 + 2 * rb) for rows, rb in points_rows)
    return n * (12 * corners + 20 * pts) + n * gather


def workload(kind, n_house):
    from draco_sharp_b200 import synth_gen as G
    if kind.startswith("c4"):
        topo = G.grid_topology(1000, 1000)
        meshes = [G.grid_mesh(1000, 1000, topo, seed=0x4000 + k) for k in range(64)]
        faces = None if kind == "c4_faces_omitted" else np.asarray(topo["corner_to_vertex"], dtype=np.uint32)
        return dict(bufs=[m[0] for m in meshes], conn=(meshes[0][1], 1000 * 1000, [topo], faces), used_maps=[topo],
                    rows=[(1000 * 1000, 12)])
    import draco_sharp_b200 as D
    house = np.fromfile(os.path.join(ROOT, "tests", "golden", "house_04.obj.drc"), dtype=np.uint8)
    bt = D.index_only([house])
    bt.host_connectivity(0)
    bt.finish()
    bi = bt.buffer_info(0)
    maps = [dict(opposite=bt.mesh_map(0, d, 0), corner_to_vertex=bt.mesh_map(0, d, 1), data_to_corner=bt.mesh_map(0, d, 2),
                 vertex_to_data=bt.mesh_map(0, d, 3)) for d in range(bi.n_attr_decoders)]
    faces = bt.faces(0)
    infos = [bt.attr_info(0, a) for a in range(bi.n_attrs)]
    used = sorted({ai.decoder_id for ai in infos})
    rb = [ai.out_bytes // ai.n_entries for ai in infos]
    bt.free()
    return dict(bufs=[house] * n_house, conn=(int(bi.attr_section_off), int(bi.n_points), maps, faces),
                used_maps=[maps[d] for d in used], rows=[(int(bi.n_points), r) for r in rb])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--house-copies", type=int, default=20000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "point_order_b200.jsonl"))
    ap.add_argument("--workloads", default="c4_faces_omitted,c4_faces_explicit,house")
    args = ap.parse_args()
    import torch
    import draco_sharp_b200 as D
    from point_order_ref import gather_rows, point_map
    if not torch.cuda.is_available():
        raise SystemExit("bench_point_order.py needs a B200: the decode path is CUDA only")
    name, power = gpu_identity()
    peak, peak_src = measured_peak()
    dec = D.DracoBatchDecoder([0])
    stream = torch.cuda.current_stream()
    dec.set_stream(0, stream.cuda_stream)
    lines = []
    rng = np.random.default_rng(20261020)
    for kind in args.workloads.split(","):
        res = workload(kind, args.house_copies)
        batches = {p: build(dec, kind, p, res) for p in (False, True)}
        outs = {}
        for p, b in batches.items():
            dec.upload(b)
            outs[p] = torch.empty(b.out_bytes, dtype=torch.uint8, device="cuda")
        ms = {False: [], True: []}
        for i in range(args.warmup + args.steps):
            for p in (False, True):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                dec.decode_resident(batches[p], dev_out=outs[p].data_ptr())
                e1.record(stream)
                torch.cuda.synchronize()
                if i >= args.warmup:
                    ms[p].append(e0.elapsed_time(e1))
        n = len(res["bufs"])
        for k in range(n):
            assert batches[True].status(k) == 0 and batches[False].status(k) == 0, k
        # seeded sample: point order == NumPy gather of the entry-order output of this run
        _, n_points, maps, faces = res["conn"]
        fl = (np.asarray(maps[0]["corner_to_vertex"]) if faces is None else np.asarray(faces)).ravel()
        checked = 0
        for k in sorted(rng.choice(n, size=min(4, n), replace=False).tolist()):
            for a in range(batches[True].buffer_info(k).n_attrs):
                ae, ap_ = batches[False].attr_info(k, a), batches[True].attr_info(k, a)
                ent = outs[False][ae.out_off: ae.out_off + ae.out_bytes].cpu().numpy()
                got = outs[True][ap_.out_off: ap_.out_off + ap_.out_bytes].cpu().numpy()
                m = maps[ae.decoder_id]
                want = gather_rows(ent, ae.out_bytes // ae.n_entries, point_map(fl, m["corner_to_vertex"], m["vertex_to_data"], n_points))
                assert np.array_equal(got, want), (kind, k, a)
                checked += 1
        # the point stage alone: torch.profiler, a separate run
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                dec.decode_resident(batches[True], dev_out=outs[True].data_ptr())
            torch.cuda.synchronize()
        stage_us = {}
        for ev in prof.key_averages():
            for kname in ("point_win_kernel", "point_resolve_kernel", "point_gather_kernel"):
                if kname in ev.key:
                    stage_us[kname] = stage_us.get(kname, 0.0) + getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0)) / 3
        stage_ms = sum(stage_us.values()) / 1e3
        gather_ms = sum(v for k2, v in stage_us.items() if "gather" in k2) / 1e3
        bytes_stage = algo_bytes(res, res["rows"])
        bytes_gather = n * sum(rows * (4 + 2 * rb) for rows, rb in res["rows"])
        # e2e, alternating
        e2e = {False: [], True: []}
        host = {p: np.empty(batches[p].out_bytes, dtype=np.uint8) for p in (False, True)}
        for i in range(args.e2e_steps + 1):
            for p in (False, True):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                b2 = build(dec, kind, p, res)
                dec.decode(b2, host_out=host[p])
                dt = (time.perf_counter() - t0) * 1e3
                b2.free()
                if i > 0:
                    e2e[p].append(dt)
        line = {
            "workload": kind, "buffers": n, "points": int(n * n_points), "gpu": name, "power_limit_and_max_sm_clock": power,
            "resident_ms_entries": float(np.median(ms[False])), "resident_ms_points": float(np.median(ms[True])),
            "resident_ms_entries_all": [round(x, 3) for x in ms[False]], "resident_ms_points_all": [round(x, 3) for x in ms[True]],
            "point_over_entry": float(np.median(ms[True]) / np.median(ms[False])),
            "point_stage_ms": stage_ms, "point_stage_kernels_us": stage_us,
            "point_stage_algo_bytes": int(bytes_stage), "point_stage_share_of_peak": (bytes_stage / (stage_ms * 1e-3) / 1e9) / peak if stage_ms else None,
            "gather_ms": gather_ms, "gather_algo_bytes": int(bytes_gather),
            "gather_share_of_peak": (bytes_gather / (gather_ms * 1e-3) / 1e9) / peak if gather_ms else None,
            "peak_gbs": peak, "peak_source": peak_src,
            "e2e_ms_entries": float(np.mean(e2e[False])), "e2e_ms_points": float(np.mean(e2e[True])),
            "out_bytes_entries": int(batches[False].out_bytes), "out_bytes_points": int(batches[True].out_bytes),
            "sample_attrs_checked": checked,
        }
        print(json.dumps(line), flush=True)
        lines.append(line)
        for b in batches.values():
            b.free()
        del outs
        torch.cuda.empty_cache()
    dec.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
