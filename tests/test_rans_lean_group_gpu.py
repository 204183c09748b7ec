"""-m gpu: the group length of the software-pipelined lean loop (DCB_LEAN_GROUP = 4 / 8 / 16 entries per group).

The switch is read once per process, so each length decodes the same batches in a child process of its own, with the
direct slot LUT off (DCB_NO_DIRECT) so that the groups run rans_raw_fused and its lean loop.  Each child checks every
batch against the oracle (statuses, and the bytes of every ok buffer) and saves them; the parent requires 8 and 16 to
give exactly what 4 gives.  The batches:
  * synthetic clouds (positions: mode 1, NCP 3; normals: mode 3, NCP 2; colours: mode 2, NCP 3) with point counts at
    every residue mod 16, short and long: how many entries the LAST group and the careful tail are left with varies
    with the count (where each lane's fast loop stops also depends on the warp it is packed into);
  * a full warp of one table in which one lane's stream needs far fewer bytes per entry than the others: its budget
    runs out first and the run budget is recomputed while the other lanes carry on;
  * truncated and bit-flipped copies of a cloud next to intact ones, and the catalogue's malformed streams;
  * the reference's sample mesh (parallelogram positions: mode 4).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import rans_cases as RC
from common import cloud
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUPS = (4, 8, 16)


def cloud_batch():
    bufs = []
    for k, base in enumerate((64, 3000, 40000)):
        for r in range(16):
            bufs.append(cloud(base + r, seed=900 + 16 * k + r, scheme=1, normal_bits=10, colors=1))
    return bufs


def short_lane_batch(num_sms):
    """Fills the machine with one table so that warps run 32 lanes; lane 5 of the first warp decodes a stream of the
    same length whose symbols are nearly all the table's widest entry (a fraction of a byte per entry)."""
    rng = np.random.default_rng(55)
    wt = RC.table_from_widths([3000] + RC.fill([], (1 << 12) - 3000, 60))
    n = 6000
    dense = RC.draw(rng, wt, 3 * n)
    skew = [0 if rng.random() < 0.995 else s for s in dense]
    full = RC.Case("lane_full", "uniform over the entries", n, [RC.pos_attr(dense, wt, 5, (0, 200))])
    short = RC.Case("lane_short", "mostly the widest entry", n, [RC.pos_attr(skew, wt, 5, (0, 200))])
    bufs = [full.buf] * (num_sms * 32)
    bufs[5] = short.buf
    return bufs


def damaged_batch():
    base = cloud(20000, seed=77, scheme=1, normal_bits=10, colors=1)
    rng = np.random.default_rng(78)
    bufs = [base]
    for keep in (0.999, 0.9, 0.6, 0.3):
        bufs.append(base[: int(len(base) * keep)].copy())
    for _ in range(8):
        b = base.copy()
        pos = int(rng.integers(len(b) // 8, len(b)))
        b[pos] ^= np.uint8(1 << int(rng.integers(0, 8)))
        bufs.append(b)
    bufs += [c.buf for c in RC.malformed()]
    return bufs + [base]


def decode_saved(dec, bufs, mesh=False):
    """Statuses and the decoded bytes of every ok buffer, in buffer order."""
    batch = dec.index(bufs)
    if mesh:
        for k in range(len(bufs)):
            batch.host_connectivity(k)
        batch.finish()
    out, _ = dec.decode(batch)
    status = np.array([batch.status(k) for k in range(len(bufs))], dtype=np.int32)
    parts = []
    for k in range(len(bufs)):
        if status[k] == 0:
            for a in range(batch.buffer_info(k).n_attrs):
                ai = batch.attr_info(k, a)
                parts.append(out[ai.out_off: ai.out_off + ai.out_bytes].copy())
    batch.free()
    return status, (np.concatenate(parts) if parts else np.zeros(0, np.uint8))


def check_oracle(bufs, status, data):
    seen = {}  # batches repeat buffer objects: decode each once
    off = 0
    for k, b in enumerate(bufs):
        o = seen.get(id(b)) or seen.setdefault(id(b), O.decode(b))
        assert status[k] == o.status, (k, status[k], o.status)
        if o.status == 0:
            for oa in o.attrs:
                got = data[off: off + oa.out.nbytes]
                assert np.array_equal(got, oa.out.view(np.uint8).ravel()), (k, "differs from the oracle")
                off += oa.out.nbytes


def test_lean_group_child(gpu_decoder):
    """The body of one group length: runs only inside the child process that test_lean_group starts."""
    dest = os.environ.get("DCB_LEAN_GROUP_OUT")
    if not dest:
        pytest.skip("runs in the child of test_lean_group")
    num_sms = __import__("torch").cuda.get_device_properties(0).multi_processor_count
    house = np.fromfile(os.path.join(ROOT, "tests", "golden", "house_04.obj.drc"), dtype=np.uint8)
    saved = {}
    for name, bufs, mesh in (("clouds", cloud_batch(), False), ("short_lane", short_lane_batch(num_sms), False),
                             ("damaged", damaged_batch(), False), ("mesh", [house] * 4, True)):
        status, data = decode_saved(gpu_decoder, bufs, mesh)
        check_oracle(bufs, status, data)
        saved[name + "_status"], saved[name + "_data"] = status, data
    assert (saved["clouds_status"] == 0).all() and (saved["short_lane_status"] == 0).all() and (saved["mesh_status"] == 0).all()
    assert (saved["damaged_status"] != 0).any()
    np.savez(dest, **saved)


@pytest.fixture(scope="module")
def by_group(tmp_path_factory):
    d = tmp_path_factory.mktemp("lean_group")
    res = {}
    for e in GROUPS:
        dest = str(d / ("e%d.npz" % e))
        env = dict(os.environ, DCB_LEAN_GROUP=str(e), DCB_NO_DIRECT="1", DCB_LEAN_GROUP_OUT=dest)
        r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                            "test_lean_group_child"], env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
        res[e] = dict(np.load(dest))
    return res


@pytest.mark.parametrize("e", [8, 16])
@pytest.mark.parametrize("batch", ["clouds", "short_lane", "damaged", "mesh"])
def test_lean_group(by_group, e, batch):
    if os.environ.get("DCB_LEAN_GROUP_OUT"):
        pytest.skip("already the child")
    ref, got = by_group[4], by_group[e]
    assert np.array_equal(got[batch + "_status"], ref[batch + "_status"])
    assert np.array_equal(got[batch + "_data"], ref[batch + "_data"])
