"""Group length of the software-pipelined lean loop (DCB_LEAN_GROUP = 4 / 8 / 16 entries per group) on configs[1].

The switch is read once per process, so every decode runs in a child process of its own: the c2 batch of bench.py
(10,000 clouds x 100,000 points, 2,048 distinct, Raw rANS), indexed and uploaded once, warm-up steps, then timed
steps between CUDA events.  The E values alternate over the rounds.  Per run the child reports the step time (events),
the Raw rANS kernel time of the library's own events (ms_raw, mean over the timed steps), the SM clock sampled under
load, cycles per symbol (ms_raw x clock / 300,000 symbols per stream), the card's name and power limit, and a
blake2b digest of the whole output arena.  The parent checks that the digests agree across E, fits
T(E) = a + b/E to the median cycles per symbol of the --fit lengths (b/E: the per-group boundary's share of a
symbol; 16 is left out by default: its unrolled body, ~2,900 SASS instructions, is slower for reasons of its own)
and writes JSON lines to stdout and to --out (default profiles/lean_group_b200.jsonl)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SYMBOLS_PER_STREAM = 100000 * 3


def gpu_identity():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = "unknown"
    return torch.cuda.get_device_name(0), q


def arena_digest(d_out, chunk=1 << 29):
    """blake2b over the digests of 512 MB slices of the device output arena (slices hashed on host threads)."""
    n = d_out.numel()
    parts = [(o, min(chunk, n - o)) for o in range(0, n, chunk)]
    with ThreadPoolExecutor(max_workers=8) as ex:
        futs = [ex.submit(lambda a: hashlib.blake2b(a).digest(), d_out[o: o + m].cpu().numpy()) for o, m in parts]
        h = hashlib.blake2b()
        for f in futs:
            h.update(f.result())
    return h.hexdigest()


def child(args):
    import torch
    import bench as B
    import draco_sharp_b200 as D
    if not torch.cuda.is_available():
        raise SystemExit("bench_lean_group.py needs a B200: the decode path is CUDA only")
    name, power = gpu_identity()
    arena, offs, lens, sums, _, _ = B.make_workload("c2", 0, 2048)
    dec = D.DracoBatchDecoder([0])
    stream = torch.cuda.current_stream()
    dec.set_stream(0, stream.cuda_stream)
    batch = dec.index_arena(arena, offs, lens)
    dec.upload(batch)
    d_out = torch.empty(batch.out_bytes, dtype=torch.uint8, device="cuda")
    sampler = B.ClockSampler(0)
    sampler.start()
    for _ in range(args.warmup):
        dec.decode_resident(batch, dev_out=d_out.data_ptr())
    torch.cuda.synchronize()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms_raw = []
    ev0.record(stream)
    for _ in range(args.steps):
        dec.decode_resident(batch, dev_out=d_out.data_ptr())
        ms_raw.append(dec.stats().ms_raw)
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    bad = sum(1 for k in range(batch.n_bufs) if batch.status(k) != 0)
    line = {"E": int(os.environ["DCB_LEAN_GROUP"]), "round": args.round, "gpu": name, "power_limit_and_max_sm_clock": power,
            "sm_mhz_under_load": clocks.get("sm_mhz"), "clock_event_reasons": clocks.get("reasons"),
            "steps": args.steps, "ms_per_step": ev0.elapsed_time(ev1) / args.steps, "ms_raw": float(np.mean(ms_raw)),
            "ms_raw_min": float(np.min(ms_raw)), "ms_raw_max": float(np.max(ms_raw)), "failed_buffers": bad}
    if clocks.get("sm_mhz"):
        line["cycles_per_symbol"] = line["ms_raw"] * 1e-3 * clocks["sm_mhz"] * 1e6 / SYMBOLS_PER_STREAM
    if args.digest:
        line["arena_blake2b"] = arena_digest(d_out)
    print("RESULT " + json.dumps(line), flush=True)
    dec.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", default="4,8,16")
    ap.add_argument("--fit", default="4,8", help="group lengths the fit T(E) = a + b/E uses")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lean_group_b200.jsonl"))
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--round", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--digest", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args)
    groups = [int(x) for x in args.groups.split(",")]
    lines = []
    for r in range(args.rounds):
        order = groups if r % 2 == 0 else groups[::-1]
        for e in order:
            cmd = [sys.executable, os.path.abspath(__file__), "--child", "--round", str(r), "--steps", str(args.steps),
                   "--warmup", str(args.warmup)] + (["--digest"] if r == 0 else [])
            t0 = time.time()
            p = subprocess.run(cmd, env=dict(os.environ, DCB_LEAN_GROUP=str(e)), stdout=subprocess.PIPE, text=True)
            res = [json.loads(x[7:]) for x in p.stdout.splitlines() if x.startswith("RESULT ")]
            if p.returncode != 0 or not res:
                raise SystemExit("child E=%d round %d failed (exit %d):\n%s" % (e, r, p.returncode, p.stdout[-3000:]))
            res[0]["child_s"] = round(time.time() - t0, 1)
            print(json.dumps(res[0]), flush=True)
            lines.append(res[0])
    digests = {l["E"]: l["arena_blake2b"] for l in lines if "arena_blake2b" in l}
    assert all(l["failed_buffers"] == 0 for l in lines), "buffers failed"
    assert len(set(digests.values())) == 1, "output arenas differ across E: %s" % digests
    med = {e: float(np.median([l["cycles_per_symbol"] for l in lines if l["E"] == e and "cycles_per_symbol" in l]))
           for e in groups}
    summary = {"summary": True, "identical_arenas_across_E": True, "gpu": lines[0]["gpu"],
               "power_limit_and_max_sm_clock": lines[0]["power_limit_and_max_sm_clock"],
               "median_cycles_per_symbol": med,
               "median_ms_raw": {e: float(np.median([l["ms_raw"] for l in lines if l["E"] == e])) for e in groups},
               "median_ms_per_step": {e: float(np.median([l["ms_per_step"] for l in lines if l["E"] == e])) for e in groups},
               "spread_ms_raw": {e: [min(l["ms_raw"] for l in lines if l["E"] == e), max(l["ms_raw"] for l in lines if l["E"] == e)]
                                 for e in groups}}
    fit = [e for e in (int(x) for x in args.fit.split(",")) if e in med]
    if len(fit) >= 2:
        # least squares T(E) = a + b/E over the medians
        A = np.array([[1.0, 1.0 / e] for e in fit])
        (a, b), *_ = np.linalg.lstsq(A, np.array([med[e] for e in fit]), rcond=None)
        summary["fit"] = {"groups": fit, "a_cycles_per_symbol": float(a), "b_cycles_per_symbol_x_entries": float(b),
                          "boundary_cycles_per_symbol_at_E4": float(b) / 4.0,
                          "what": "T(E) = a + b/E; b/E is the share of one symbol in the cost of a group boundary"}
    print(json.dumps(summary), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for l in lines + [summary]:
            f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
