"""-m gpu: the rANS table catalogue (rans_cases.py) through the C ABI, under every kernel-selection switch.

Every case decodes three times (plain: the lean / software-pipelined instantiations; DCB_DUMP_SYMBOLS; DCB_DUMP_QINTS)
and must give the symbols it encoded (malformed ones: what rans_ref decodes), the quantised ints of a Python delta +
wrap, the oracle's output bytes and the oracle's status.  The switches are read once per process, so every variant
runs in a child process with DCB_DEBUG_PLAN=1; the child parses the plan lines and fails when a group that should
have taken the variant's kernel went to another one.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import rans_cases as RC
import rans_ref as R
from common import compare_with_oracle, gpu_decode_all
from draco_sharp_b200 import _native as N
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu

_ND = {"DCB_NO_DIRECT": "1"}
VARIANTS = {
    "default": {},
    "no_direct": dict(_ND),
    "no_split": dict(_ND, DCB_NO_SPLIT="1"),
    "no_lean": dict(_ND, DCB_NO_LEAN="1"),
    "lutb_full": dict(_ND, DCB_LUTB_FULL="1"),
    **{"rec_ka%d" % k: dict(_ND, DCB_REC="1", DCB_REC_KA=str(k)) for k in range(RC.REC_KA0, RC.REC_KA0 + 4)},
    "pc": dict(_ND, DCB_RANS_PC="1"),
    "pc_no_fused": dict(_ND, DCB_RANS_PC="1", DCB_NO_PC_FUSED="1"),
    "split_rec": dict(_ND, DCB_REC="1", DCB_SPLIT="1"),
    "split_pc": dict(_ND, DCB_RANS_PC="1", DCB_SPLIT="1"),
    "no_fast_tagged": {"DCB_NO_FAST_TAGGED": "1"},
}
_PLAN = re.compile(r"\[dcb plan\] (raw|tag) group (.*)")


def plan_lines(err):
    out = []
    for m in _PLAN.finditer(err):
        f = {k: int(v) for k, v in re.findall(r"(\w+)=(-?\d+)", m.group(2))}
        f["kind"] = m.group(1)
        f["streams"] = int(re.search(r"(\d+) streams", m.group(2)).group(1))
        out.append(f)
    return out


def check_case(dec, case):
    """Decode the case alone three times and check it."""
    gpu = gpu_decode_all(dec, [case.buf])
    compare_with_oracle(gpu, [case.buf])
    check_result(case, gpu[0])


def check_result(case, g):
    """One buffer's GPU results (gpu_decode_all) against the symbols the case encoded, or what rans_ref decodes."""
    ref, status = case.reference()
    assert g["status"] == status, (case.name, g["status"], status)
    if status != R.OK:
        return
    for a, (st, syms), ga in zip(case.attrs, ref, g["attrs"]):
        want = a.symbols if case.valid else syms
        assert np.array_equal(ga["symbols"].view(np.uint32), np.asarray(want, dtype=np.uint32)), (case.name, a.kind)
        assert np.array_equal(ga["qints"], np.asarray(a.qints(want), dtype=np.int32)), (case.name, a.kind)


def rec_shape(case, ka):
    return case.prob is not None and case.prec <= 15 and ka < case.prec and RC.rec_cuts(case.prob, ka) is not None


def check_plan(variant, case, lines):
    """The groups of a one-case batch took the variant's kernel."""
    has_tag = any(a.kind == "tag" for a in case.attrs)
    if case.valid and has_tag:
        assert any(f["kind"] == "tag" for f in lines), (variant, case.name)
    e = getattr(case, "expect", {})
    for f in lines:
        small = f["wide"] == 0 if "wide" in f else True
        u16 = small and not f["global"]
        if f["kind"] == "raw" and case.plan:
            for k, v in case.plan.items():
                assert f[k] == v, (variant, case.name, k, f)
        # the two-level kernels: the two-region LUT splits at the case's kA; the dense table's probe searches
        two_level = f["kind"] == "raw" and u16 and variant in ("no_direct", "no_lean", "lutb_full")
        if two_level and "split_k" in e:
            assert RC.split_choice(case.prob, case.prec, f["lut"], f["lutb"]) == e["split_k"], (variant, case.name, f)
        if f["kind"] == "raw" and u16 and not f["direct"] and not f["rec_ka"] and e.get("search"):
            assert RC.search_hit(case.prob, 1 << f["k"], f["compact"] == 1), (variant, case.name, f)
        if variant == "default":
            if u16 and f["prec"] <= 13:
                assert f["direct"] == 1, (variant, case.name, f)
        elif variant in ("no_direct", "no_split", "no_lean", "lutb_full"):
            assert f["direct"] == 0 and f["pairs"] == 0 and f["rec_ka"] == 0, (variant, case.name, f)
            if u16 and f["compact"]:
                assert f["lutb"] > 0, (variant, case.name, f)
        elif variant.startswith("rec_ka"):
            ka = int(variant[6:])
            assert f["direct"] == 0 and f["rec_ka"] in (0, ka), (variant, case.name, f)
            if case.prob is not None:  # the table of every group of the case (tag groups: a precision-12 tag table)
                want = ka if u16 and rec_shape(case, ka) else 0
                assert f["rec_ka"] == want, (variant, case.name, want, f)
                if want:
                    assert f["pairs"] > 0 and f["rec"] == RC.rec_bytes(case.prob, ka), (variant, case.name, f)
        elif variant in ("pc", "pc_no_fused"):
            if u16:
                assert f["pairs"] > 0 and f["direct"] == 0 and f["rec_ka"] == 0, (variant, case.name, f)
        elif variant == "split_rec":
            if case.prob is not None:
                shaped = u16 and any(rec_shape(case, k) for k in range(RC.REC_KA0, RC.REC_KA0 + 4))
                assert (f["rec_ka"] > 0) == shaped, (variant, case.name, f)
                if shaped:
                    assert f["split"] == 1 and rec_shape(case, f["rec_ka"]), (variant, case.name, f)
        elif variant == "split_pc":
            if u16:
                assert f["pairs"] > 0, (variant, case.name, f)
                if f["prec"] <= 12 and f["kind"] == "raw":
                    assert f["split"] == 1, (variant, case.name, f)


def run_variant(variant, dec, capfd):
    num_sms = __import__("torch").cuda.get_device_properties(0).multi_processor_count
    cases = [c for c in RC.catalogue() + RC.malformed() if variant == "default" or not c.long]
    if variant == "no_fast_tagged":
        cases = [c for c in cases if any(a.kind == "tag" for a in c.attrs)]
    took = {}
    capfd.readouterr()
    for c in cases:
        check_case(dec, c)
        lines = plan_lines(capfd.readouterr().err)
        check_plan(variant, c, lines)
        for f in lines:
            for k in ("direct", "rec_ka", "pairs", "split", "global", "lutb"):
                took[k] = took.get(k, 0) + (f[k] > 0)
    # the variant's kernel ran at all
    need = {"default": ("direct", "global"), "no_direct": ("lutb",), "lutb_full": ("lutb",), "pc": ("pairs",),
            "pc_no_fused": ("pairs",), "split_rec": ("rec_ka", "split"), "split_pc": ("pairs", "split")}
    for k in need.get(variant, ("rec_ka",) if variant.startswith("rec_ka") else ()):
        assert took.get(k, 0) > 0, (variant, k, took)
    if variant.startswith("rec_ka"):
        # the record tables nearest the shared-memory limit: the largest the planner accepts runs on the record
        # kernels with exactly the table area the Python layout gives, the next larger one is refused
        acc, ref = RC.rec_limit(num_sms, int(variant[6:]))
        for c, want in ((acc, int(variant[6:])), (ref, 0)):
            lines = check_copies(dec, c, capfd)
            assert len(lines) == 1 and lines[0]["rec_ka"] == want, (c.name, lines)
            if want:
                f = lines[0]
                assert (f["lanes"], f["pairs"], f["rec"]) == (4, 4, c.rec_bytes), (c.name, f)
    if variant == "no_direct":
        # a compact table whose two-region LUT does not fit beside 8 streams per SM: the uniform LUT with its search
        c = RC.no_split(num_sms)
        lines = check_copies(dec, c, capfd)
        assert len(lines) == 1, lines
        f = lines[0]
        assert f["rec_ka"] == 0 and f["direct"] == 0 and f["pairs"] == 0 and f["compact"] == 1, f
        assert RC.split_choice(c.prob, c.prec, f["lut"], f["lutb"]) is None, f
        assert RC.search_hit(c.prob, 1 << f["k"], True), f
    if variant != "default":
        return
    # the whole catalogue in one batch: groups of mixed shapes, long streams
    bufs = [c.buf for c in cases]
    gpu = gpu_decode_all(dec, bufs)
    assert compare_with_oracle(gpu, bufs) == sum(1 for c in cases if c.reference()[1] == R.OK)
    for c, g in zip(cases, gpu):
        check_result(c, g)
    # the catalogue next to a machine-filling group of tiny clouds: its groups lose the direct slot LUT
    tiny = RC.Case("tiny", "tiny cloud", 2, [RC.pos_attr([1, 2, 3, 0, 1, 2], [1024] * 4, 5, (-9, 9))])
    bufs = [c.buf for c in cases] + [tiny.buf] * (num_sms * 8)
    capfd.readouterr()
    gpu = gpu_decode_all(dec, bufs)
    lines = plan_lines(capfd.readouterr().err)
    assert compare_with_oracle(gpu, bufs) == len(bufs) - sum(1 for c in cases if c.reference()[1] != R.OK)
    for c, g in zip(cases, gpu):
        check_result(c, g)
    assert any(f["kind"] == "raw" and f["streams"] >= num_sms * 8 for f in lines), lines
    for f in lines:
        if f["kind"] == "raw" and f["streams"] < num_sms * 8:  # tag groups are planned on their own
            assert f["direct"] == 0, f
    # one warp, 31 lean-eligible streams and one that is not
    bufs, odd_at, lean, odd = RC.warp_mix(num_sms)
    batch = dec.index(bufs)
    capfd.readouterr()
    out, _ = dec.decode(batch)
    lines = [f for f in plan_lines(capfd.readouterr().err) if f["kind"] == "raw"]
    assert len(lines) == 1 and lines[0]["lanes"] == 32 and lines[0]["direct"] == 0, lines
    want = {k: O.decode(c.buf).attrs[0].out for k, c in (("lean", lean), ("odd", odd))}
    for k in range(len(bufs)):
        ai = batch.attr_info(k, 0)
        assert batch.status(k) == 0
        assert np.array_equal(out[ai.out_off: ai.out_off + ai.out_bytes], want["odd" if k == odd_at else "lean"]), k
    batch.free()


def check_copies(dec, case, capfd):
    """Decode case.n_bufs copies of the case's buffer (plain and DUMP_SYMBOLS); every copy gives the case's bytes and
    symbols.  Returns the decode's raw plan lines."""
    bufs = [case.buf] * case.n_bufs
    want = O.decode(case.buf).attrs[0].out
    syms = np.asarray(case.attrs[0].symbols, dtype=np.uint32)
    capfd.readouterr()
    for flags in (0, N.DCB_DUMP_SYMBOLS):
        batch = dec.index(bufs)
        out, dbg = dec.decode(batch, flags=flags)
        for k in range(len(bufs)):
            assert batch.status(k) == 0, (case.name, k, batch.status(k))
            ai = batch.attr_info(k, 0)
            if flags:
                assert np.array_equal(dbg[ai.dbg_off: ai.dbg_off + 4 * syms.size].view(np.uint32), syms), (case.name, k)
            else:
                assert np.array_equal(out[ai.out_off: ai.out_off + ai.out_bytes], want), (case.name, k)
        batch.free()
    return [f for f in plan_lines(capfd.readouterr().err) if f["kind"] == "raw"][:1]


def test_variant_child(gpu_decoder, capfd):
    """The body of one variant: runs only inside the child process that test_variant starts."""
    variant = os.environ.get("DCB_TABLES_VARIANT")
    if not variant:
        pytest.skip("runs in the child of test_variant")
    run_variant(variant, gpu_decoder, capfd)


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variant(variant):
    if os.environ.get("DCB_TABLES_VARIANT"):
        pytest.skip("already the child")
    env = dict(os.environ, DCB_TABLES_VARIANT=variant, DCB_DEBUG_PLAN="1", **VARIANTS[variant])
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", "test_variant_child"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "1 passed" in r.stdout
