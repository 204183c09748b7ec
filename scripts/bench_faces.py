"""Faces in the output arena (DCB_FACES_ARENA, DESIGN.md 3.6c): what the mode costs and saves against today's path.

Workloads (sequential meshes are written by tests/drc_writer.py, one distinct mesh per workload, repeated in the batch):
  raw      --grids grids of --side x --side vertices, index differences in the Raw scheme (method 0)
  varint   the same grids with plain varint indices (method 1, 65536 <= points < 2^21)
  small    --small meshes of 41 x 41 vertices (1,681 points, Raw indices, one quantized position attribute)
  house    --houses copies of the reference's sample (Edgebreaker), point order, with and without the mode
For each workload and each mode (off: dcb_host_connectivity decodes the indices; on: it locates them, the GPU decodes):
  host_ms    wall time of the dcb_host_connectivity loop
  step_ms    dcb_decode_resident of the uploaded batch (median of --steps, each ending in a synchronise)
  e2e_ms     index + connectivity + finish + dcb_decode (H2D, kernels, D2H), one call
  kernels    device time per kernel name from torch.profiler (a separate pass), with the index chain's bound (DESIGN 3.1:
             symbols per stream x cycles per symbol / clock) and the scan / plain kernels' algorithmic bytes over the time
One JSON line per (workload, mode) goes to --out, the first line records the card's name, power limit and clock.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import draco_sharp_b200 as D  # noqa: E402
import drc_writer as W  # noqa: E402
import faces_ref as F  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
CYCLES_PER_SYMBOL = 95.0  # c4's direct-LUT Raw chain (DESIGN 3.1): the estimate the bound uses


def gpu_card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_mhz": float(clock)}


def build_batch(dec, bufs, faces, points):
    t0 = time.perf_counter()
    b = dec.index(bufs)
    if points:
        b.set_output_order(True)
    if faces:
        b.set_face_output(True)
    t1 = time.perf_counter()
    for k in range(len(bufs)):
        if b.buffer_info(k).needs_connectivity:
            b.host_connectivity(k)
    t2 = time.perf_counter()
    b.finish()
    return b, (t2 - t1) * 1e3, (t1 - t0) * 1e3


def profile_kernels(dec, batch):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dec.decode_resident(batch)
        torch.cuda.synchronize()
    ms = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            m = re.search(r"(\w+)\s*[<(]", e.name.replace("(anonymous namespace)::", "").replace("void ", "", 1))
            key = m.group(1) if m else e.name.strip()
            ms[key] = ms.get(key, 0.0) + e.device_time / 1e3
    return ms


def run(dec, name, bufs, points, steps, card, seq_info):
    rows = []
    for faces in (False, True):
        t0 = time.perf_counter()
        batch, host_ms, _ = build_batch(dec, bufs, faces, points)
        out, _ = dec.decode(batch)
        e2e_ms = (time.perf_counter() - t0) * 1e3
        assert all(batch.status(k) == 0 for k in range(len(bufs)))
        d2h = batch.out_bytes
        batch.free()
        batch, _, _ = build_batch(dec, bufs, faces, points)
        dec.upload(batch)
        dec.decode_resident(batch)
        t = []
        for _ in range(steps):
            s = time.perf_counter()
            dec.decode_resident(batch)
            t.append((time.perf_counter() - s) * 1e3)
        kern = profile_kernels(dec, batch)
        row = {"workload": name, "faces_in_arena": faces, "buffers": len(bufs), "host_ms": round(host_ms, 2),
               "step_ms": round(float(np.median(t)), 3), "e2e_ms": round(e2e_ms, 1), "out_bytes": d2h,
               "kernels_ms": {k: round(v, 3) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])[:8]}}
        if faces and seq_info:
            n_idx, width = seq_info
            total_idx = n_idx * len(bufs)
            if width < 0:  # Raw: the chain bound of one stream, and the scan's algorithmic bytes (4 B in + 4 B out per index)
                row["chain_bound_ms"] = round(n_idx * CYCLES_PER_SYMBOL / (card["max_sm_mhz"] * 1e3), 2)
                scan = sum(v for k, v in kern.items() if k.startswith("seq_index"))
                if scan:
                    row["scan_ms"] = round(scan, 3)
                    row["scan_hbm_share"] = round(8 * total_idx / (scan / 1e3) / HBM_BYTES_PER_S, 3)
            else:  # plain: width (varint: its bytes) + 4 B per index
                k = "seq_varint_kernel" if width == 0 else "seq_plain_kernel"
                in_bytes = sum(len(b) for b in bufs) if width == 0 else width * total_idx
                if kern.get(k):
                    row["plain_ms"] = round(kern[k], 3)
                    row["plain_hbm_share"] = round((in_bytes + 4 * total_idx) / (kern[k] / 1e3) / HBM_BYTES_PER_S, 3)
        rows.append(row)
        batch.free()
        print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, default=64)
    ap.add_argument("--side", type=int, default=1000)
    ap.add_argument("--small", type=int, default=20000)
    ap.add_argument("--houses", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default="raw,varint,small,house")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    card = gpu_card()
    dec = D.DracoBatchDecoder()
    n_pts = a.side * a.side
    faces = F.grid_faces(a.side, a.side)
    rows = [dict(card, kind="card")]
    for w in a.workloads.split(","):
        if w == "raw":
            m = F.mesh(faces, n_pts, 0, "raw", with_attrs=False)
            rows += run(dec, w, [m] * a.grids, False, a.steps, card, (3 * len(faces), -1))
        elif w == "varint":
            m = F.mesh(faces, n_pts, 1, with_attrs=False)
            rows += run(dec, w, [m] * a.grids, False, a.steps, card, (3 * len(faces), F.index_width(n_pts)))
        elif w == "small":
            m = F.mesh(F.grid_faces(41, 41), 41 * 41, 0, "raw", seed=5)
            rows += run(dec, w, [m] * a.small, False, a.steps, card, (3 * 2 * 40 * 40, -1))
        elif w == "house":
            h = np.fromfile(os.path.join(ROOT, "tests", "golden", "house_04.obj.drc"), dtype=np.uint8)
            rows += run(dec, w, [h] * a.houses, True, a.steps, card, None)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
