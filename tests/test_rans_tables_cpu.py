"""-m "not gpu": the rANS table catalogue (rans_cases.py) on the CPU.  Every valid case decodes to the symbols it
encoded, through the plain reference restatement (rans_ref.py) and through the oracle; every malformed case gives
the same status and symbols from both; and each case's table has the feature it claims."""
import ctypes as C

import numpy as np
import pytest

import drc_writer as W
import rans_cases as RC
import rans_ref as R
from oracle import pyoracle as O


@pytest.fixture(scope="module")
def cases():
    return RC.catalogue()


@pytest.fixture(scope="module")
def bad_cases():
    return RC.malformed()


def test_catalogue_covers_its_features(cases):
    names = [c.name for c in cases]
    assert len(set(names)) == len(names)
    for c in cases:
        e = getattr(c, "expect", {})
        prob = c.prob
        if "first_narrow" in e:
            ka, slot = e["first_narrow"]
            assert RC.first_narrow(prob, ka) == slot, c.name
            na = sum(1 for p in prob if p)
            assert 2 * na + 1 < len(prob), c.name  # compact: the only tables the two-region LUT is built for
        if "compact" in e:
            na = sum(1 for p in prob if p)
            assert (2 * na + 1 < len(prob)) == e["compact"], c.name
        if e.get("dense"):
            na = sum(1 for p in prob if p)
            assert 2 * na + 1 >= len(prob), c.name
            assert any(p == 0 for p in prob[:len(prob) - 1]), c.name  # zero-width entries between owners
        if "split_k" in e:
            # with room for every split, the device picks the case's kA (the GPU test checks it with the plan's bytes)
            P = 1 << c.prec
            assert RC.split_choice(prob, c.prec, P >> 4, P >> 1) == e["split_k"], c.name
        if "search" in e:
            # every bucket size the planner may give a dense u16 table (2^1 .. 2^(prec - 4) slots)
            assert all(RC.search_hit(prob, 1 << k, False) for k in range(1, c.prec - 3)), c.name
        if "dprefix" in e:
            d = next((i for i, (s, _, _) in enumerate(RC.entries(prob)) if s != i), sum(1 for p in prob if p))
            assert d == e["dprefix"], c.name
        if "rec" in e:
            shaped = [RC.rec_cuts(prob, ka) is not None for ka in range(RC.REC_KA0, RC.REC_KA0 + 4)]
            assert all(shaped) if e["rec"] else not any(shaped), c.name
            if e["rec"]:
                ta, tb, tc = RC.rec_cuts(prob, RC.REC_KA0)
                starts = {s for _, s, _ in RC.entries(prob)}
                assert tc in starts and max(w for _, s, w in RC.entries(prob) if s + w > tc) == 16, c.name
        if "rec_edge" in e:
            for ka in range(RC.REC_KA0, RC.REC_KA0 + 4):
                cut = RC.rec_cuts(prob, ka)[e["rec_edge"]]
                starts = {s for _, s, _ in RC.entries(prob)}
                assert cut in starts and cut + 1 in starts, c.name
        if "rec_cuts" in e:
            ta, tb, tc = RC.rec_cuts(prob, e["rec_cuts"])
            assert 0 < ta < tb < tc < (1 << c.prec), (c.name, ta, tb, tc)
        if "wide" in e:
            assert (len(prob) > 65535) == e["wide"], c.name
    # the init tags 0..3, every payload offset residue mod 16, payload lengths around the 128-byte ring
    res = set()
    for c in cases:
        if c.name.startswith("offset_pad"):
            st, _, end, _ = R.decode_symbols(c.buf, c.sym_offs[0], 3 * c.n, 3)
            pay_len = len(W.rans_payload(c.attrs[0].symbols, [256] * 16, 12))
            res.add((end - pay_len) % 16)
    assert res == set(range(16))


def test_record_limit_and_no_split_tables():
    for ka in range(RC.REC_KA0, RC.REC_KA0 + 4):
        acc, ref = RC.rec_limit(148, ka)
        assert RC.rec_fits(4, 4, acc.rec_bytes, 12) and not RC.rec_fits(4, 4, ref.rec_bytes, 12)
        assert ref.rec_bytes > acc.rec_bytes
        for c in (acc, ref):
            assert O.decode(c.buf).status == 0 and c.reference()[0][0][1] == c.attrs[0].symbols
    c = RC.no_split(148)
    assert 2 * sum(1 for p in c.prob if p) + 1 < len(c.prob)
    assert RC.split_choice(c.prob, 15, 1 << 11, (1 << 14) - 16) is None
    assert RC.search_hit(c.prob, 1 << 5, True)


def _init_tag_of(c):
    a = c.attrs[0]
    return a.field[-1] >> 6


def test_init_tags(cases):
    got = {_init_tag_of(c) for c in cases if c.name.startswith("init_tag")}
    assert got == {0, 1, 2, 3}


def test_valid_cases_decode_to_the_encoded_symbols(cases):
    for c in cases:
        ref, status = c.reference()
        assert status == R.OK, c.name
        o = O.decode(c.buf)
        assert o.status == 0, (c.name, o.status)
        assert o.n_attrs == len(c.attrs)
        for a, (st, syms), oa in zip(c.attrs, ref, o.attrs):
            assert syms == a.symbols, c.name
            assert np.array_equal(oa.symbols, np.asarray(a.symbols, dtype=np.uint32)), c.name
            assert np.array_equal(oa.qints, np.asarray(a.qints(a.symbols), dtype=np.int32)), c.name


def _oracle_symbols(buf, pos, nv, nc):
    a = np.frombuffer(bytes(buf), dtype=np.uint8)
    out = np.zeros(max(1, nv), dtype=np.uint32)
    p = C.c_uint64(pos)
    st = O.lib().orc_decode_symbols(a.ctypes.data, a.size, C.byref(p), nv, nc, out.ctypes.data, None)
    return st, out[:nv]


def test_malformed_cases_reference_and_oracle_agree(bad_cases):
    seen = set()
    for c in bad_cases:
        ref, status = c.reference()
        seen.add(status)
        for a, off, (st, syms) in zip(c.attrs, c.sym_offs, ref):
            ost, osyms = _oracle_symbols(c.buf, off, c.n * a.nc, a.nc)
            assert ost == st, (c.name, ost, st)
            if st == R.OK:
                assert np.array_equal(osyms, np.asarray(syms, dtype=np.uint32)), c.name
        o = O.decode(c.buf)
        assert o.status == status, (c.name, o.status, status)
        if status == R.OK:
            for a, (st, syms), oa in zip(c.attrs, ref, o.attrs):
                assert np.array_equal(oa.symbols, np.asarray(syms, dtype=np.uint32)), c.name
                assert np.array_equal(oa.qints, np.asarray(a.qints(syms), dtype=np.int32)), c.name
    # every failure the catalogue means to reach, and decodes that run out of bytes and still succeed
    assert {R.OK, R.TABLE, R.RANS_INIT, R.TAG, R.EOF, R.NUM_SYMBOLS} <= seen


def test_cut_payloads_decode_other_symbols(bad_cases):
    """A payload cut short decodes (status OK) to symbols other than the encoded ones: the cases test garbage that
    is defined by the reference, not a decode that happens to succeed."""
    for c in bad_cases:
        if c.name.startswith("cut_pos") and int(c.name.split("_")[-1]) >= 40:
            ref, status = c.reference()
            assert status == R.OK and ref[0][1] != c.attrs[0].symbols, c.name
