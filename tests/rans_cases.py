"""Catalogue of Raw / Tagged rANS table shapes for the conformance suite (test_rans_tables_cpu.py, _gpu.py).

Every case is a .drc point cloud whose probability tables the case chooses (drc_writer.symbols_raw_table /
symbols_tagged_table), with the symbols it encoded and the values a plain Python decode gives.  The table shapes
are the ones the kernels handle with code of their own (dcb_device.cuh RansLane::build / fill_lut, dcb_rans_rec.cu,
dcb_walk.h): the feature a case is meant to hit is computed from its table here and asserted by the CPU test.
"""
import numpy as np

import drc_writer as W
import rans_ref as R

MBL = {12: 5, 13: 9, 15: 10, 16: 11, 18: 12, 19: 13, 20: 14}  # a max_bit_length giving each precision
REC_KA0 = 5


def zz_dec(s):
    s = int(s)
    return (s >> 1) if s % 2 == 0 else -((s + 1) >> 1)


def i32(v):
    return ((int(v) + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


def delta_wrap(corr, nc, mn, mx):
    """PredictionSchemeDeltaDecoder + wrap transform (wrap_original) with Python integers and int32 wrap-around."""
    md = i32(1 + mx - mn)
    out = []
    for i, c in enumerate(corr):
        pred = 0 if i < nc else out[i - nc]
        pred = min(max(pred, mn), mx)
        o = i32(pred + c)
        if o > mx:
            o = i32(o - md)
        elif o < mn:
            o = i32(o + md)
        out.append(o)
    return out


# ---- table geometry, restated from the device code ----
def entries(prob):
    """(symbol id, start slot, width) of every entry with a non-zero probability, in table order."""
    out, c = [], 0
    for s, p in enumerate(prob):
        if p:
            out.append((s, c, int(p)))
            c += int(p)
    return out


def first_narrow(prob, ka):
    """First slot owned by an entry narrower than 2^ka (RansLane::build); 2^prec when there is none."""
    for _, start, w in entries(prob):
        if w < (1 << ka):
            return start
    return sum(int(p) for p in prob)


def rec_cuts(prob, ka):
    """RecShape (dcb_internal.h): the cuts (ta, tb, tc) for wide-region buckets of 2^ka slots, or None when the table
    does not have the bucket-record shape."""
    P = sum(int(p) for p in prob)
    scales = [3, 4] + [REC_KA0 + j for j in range(4)]
    bad, prev, end_wide = [None] * 6, [None] * 6, 0
    for _, start, w in entries(prob):
        if w > 16:
            end_wide = start + w
        if start == 0:
            continue
        for j, k in enumerate(scales):
            if start % (1 << k) == 0:
                continue
            if start >> k == prev[j] and bad[j] is None:
                bad[j] = start
            prev[j] = start >> k
    tc = bad[0] if bad[0] is not None and bad[0] < P else P
    if tc < end_wide:
        return None
    tb = min(bad[1], tc) if bad[1] is not None else tc
    fa = bad[ka - REC_KA0 + 2]
    ta = min(fa, tb) if fa is not None else tb
    return ta, tb, tc


def rec_layout_bytes(ta, tb, tc, prec, ka):
    """dcb_rec_layout(...).bytes: the table area of one lane of the bucket-record kernels."""
    n_a = (ta + (1 << ka) - 1) >> ka
    n_b = ((tb + 15) >> 4) - (ta >> 4) if tb > ta else 0
    n_b2 = ((tc + 7) >> 3) - (tb >> 3) if tc > tb else 0
    n_c = prec - tc
    off_bm = (8 * (n_a + n_b + n_b2) + n_c + 3) & ~3
    words = (n_c + 31) >> 5
    return (off_bm + 4 * words + 2 * words + 7) & ~7


def rec_bytes(prob, ka):
    """What the planner reserves per lane for this table on the record kernels (plan line `rec=`): its layout plus a
    u16 value slot per entry behind the dense prefix.  None: the table does not have the shape."""
    cuts = rec_cuts(prob, ka)
    if cuts is None:
        return None
    ent = entries(prob)
    dprefix = next((i for i, (s, _, _) in enumerate(ent) if s != i), len(ent))
    return rec_layout_bytes(*cuts, sum(int(p) for p in prob), ka) + ((2 * (len(ent) - dprefix) + 7) & ~7)


# shared memory of the record kernels (dcb_api.cu kSmemPerSM / kSmemPerCtaReserve, dcb_kernels.h DCB_REC_*,
# dcb_rans_rec.cu rec_geom): a CTA of `pairs` slices of `lanes` table areas, rings, queue, control and hand-over records
SMEM_PER_SM, CTA_RESERVE = 227 * 1024, 1024


def rec_cta_bytes(lanes, pairs, area, syms_per_group):
    o = (lanes * ((area + 7) & ~7) + 127) & ~127
    o += lanes * 128 + 2 * syms_per_group * 64 + 64 + lanes * 56
    return ((o + 127) & ~127) * max(1, pairs) + 128


def rec_fits(lanes, pairs, area, syms_per_group):
    """plan_rans_groups' test for one CTA per SM on the record kernels (one device, no co-running kernels)."""
    return rec_cta_bytes(lanes, pairs, area, syms_per_group) + CTA_RESERVE <= SMEM_PER_SM + 1024


def split_choice(prob, prec, lut_bytes, lutb_bytes):
    """The bucket size 2^kA RansLane::build picks for the two-region LUT of a compact table with `lut_bytes` of wide
    region and `lutb_bytes` of narrow region per lane: the feasible kA needing the fewest bytes.  None: no split fits,
    the uniform LUT is taken."""
    P = 1 << prec
    ent = entries(prob)
    best, best_k = None, None
    for k in range(1, 8):
        if k + 7 > prec:
            continue
        t = next((st for _, st, w in ent if w < (1 << k)), P) & ~127
        na, nbk = t >> k, (P - t) >> 1
        if na > lut_bytes or nbk > lutb_bytes:
            continue
        if best is None or na + nbk < best:
            best, best_k = na + nbk, k
    return best_k


def search_hit(prob, bucket, compact):
    """Whether the uniform LUT's probe runs its search loop for some slot: the bucket's first entry i has
    cum[i + 2] inside the bucket (compact tables hold the active entries only, dense ones every symbol)."""
    widths = [int(p) for p in prob if p] if compact else [int(p) for p in prob]
    cum = np.concatenate([[0], np.cumsum(widths)])
    P = int(cum[-1])
    cum = np.concatenate([cum, [P, P]])
    for b in range(P // bucket):
        i = int(np.searchsorted(cum, b * bucket, side="right")) - 1
        while cum[i + 1] <= b * bucket:
            i += 1
        if cum[i + 2] <= (b + 1) * bucket - 1:
            return True
    return False


def split_at(prob, slot):
    """The table with the entry that owns `slot` cut in two there (a new entry boundary at `slot`)."""
    out, c = [], 0
    for p in prob:
        if p and c < slot < c + p:
            out += [slot - c, c + p - slot]
        else:
            out.append(p)
        c += p
    return out


def table_from_widths(widths, gap=0, lead=0, tail=0):
    """Entries of the given widths in slot order; `gap` zero-probability symbols between two entries, `lead` before
    the first, `tail` behind the last."""
    prob = [0] * lead
    for i, w in enumerate(widths):
        if i:
            prob += [0] * gap
        prob.append(int(w))
    return prob + [0] * tail


def fill(widths, total, w):
    """Append entries of width w (the last one takes the rest, at most w) until the widths sum to total."""
    widths = list(widths)
    rest = total - sum(widths)
    assert rest >= 0
    while rest > 0:
        widths.append(min(w, rest))
        rest -= widths[-1]
    return widths


def random_table(rng, prec, n_active, gap=0):
    P = 1 << prec
    cuts = np.sort(rng.choice(np.arange(1, P), size=n_active - 1, replace=False))
    widths = np.diff(np.concatenate([[0], cuts, [P]]))
    return table_from_widths(widths, gap)


def final_state_for(target, sym, prob, prec):
    """An encoder start state (= the decoder's final state) that makes the encoder's last state `target` when the
    stream is the single symbol `sym`: picks the init tag of a one-symbol stream."""
    P, L = 1 << prec, 4 << prec
    cum, p = sum(int(x) for x in prob[:sym]), int(prob[sym])
    t = target - cum
    assert t % P < p
    pre = (t // P) * p + t % P
    assert 4 * p <= pre < 1024 * p
    fs = pre if pre >= L else pre * 256 + 0x5A
    assert L <= fs < 256 * L and (fs >= 1024 * p) == (pre < L)
    return fs


# ---- buffers ----
def _attr(att_type, data_type, nc, seq_type, portable, xform=b"", uid=0):
    return dict(att_type=att_type, data_type=data_type, nc=nc, seq_type=seq_type, portable=portable, xform=xform, unique_id=uid)


class Attr:
    """One attribute of a case: its bytes and what a decode of them must give."""

    def __init__(self, kind, nc, field, pred, wrap, symbols):
        self.kind, self.nc, self.field, self.wrap = kind, nc, field, wrap
        self.symbols = symbols          # the symbols the field encodes (Raw: symbol ids; Tagged: the bit-field values)
        head = bytes([pred & 0xFF]) + (bytes([1]) if pred != -2 else b"")
        self.portable = head + bytes([1]) + field + (W.wrap_data(*wrap) if wrap else b"")
        self.sym_at = len(head) + 1     # offset of the SYMBOLS field inside the portable bytes

    def qints(self, symbols):
        corr = [zz_dec(s) for s in symbols]
        return delta_wrap(corr, self.nc, *self.wrap) if self.wrap else [i32(c) for c in corr]


def pos_attr(symbols, prob, mbl, wrap, final_state=None, pad=0, field=None):
    """3-component quantised position, delta + wrap, dequantised (the kernels' mode 1)."""
    if field is None:
        field = W.symbols_raw_table(symbols, prob, mbl, final_state, pad)
    return Attr("pos", 3, field, 0, wrap, list(symbols))


def quant_attr(nc, symbols, prob, mbl, wrap, field=None):
    if field is None:
        field = W.symbols_raw_table(symbols, prob, mbl)
    return Attr("quant%d" % nc, nc, field, 0, wrap, list(symbols))


def int_attr(symbols, prob, mbl, final_state=None, pad=0, field=None):
    """1-component int32 attribute without prediction: values = zig-zag decoded symbols (the generic mode 0)."""
    if field is None:
        field = W.symbols_raw_table(symbols, prob, mbl, final_state, pad)
    return Attr("int", 1, field, -2, None, list(symbols))


def tag_attr(values, nc, tag_prob, tags, field=None):
    """Tagged int32 attribute without prediction, last in its buffer: its bit area ends where the buffer ends."""
    if field is None:
        field = W.symbols_tagged_table(values, nc, tag_prob, tags)
    return Attr("tag", nc, field, -2, None, list(values))


def build(n, attrs):
    """The .drc buffer, and per attribute the offset of its SYMBOLS field in it."""
    descs = []
    for i, a in enumerate(attrs):
        if a.kind == "tag" or a.kind == "int":
            descs.append(_attr(4, 5, a.nc, 1, a.portable, b"", i))
        else:
            descs.append(_attr(0 if a.kind == "pos" else 4, 9, a.nc, 2, a.portable, W.quant_params([0.5] * a.nc, 3.0, 20), i))
    buf = W.point_cloud(n, descs)
    tail = sum(len(d["xform"]) for d in descs)
    offs = []
    for i, a in enumerate(attrs):
        offs.append(len(buf) - tail - sum(len(d["portable"]) for d in descs[i:]) + a.sym_at)
    return buf, offs


class Case:
    def __init__(self, name, feature, n, attrs, long=False, prob=None, prec=None, plan=None, mutate=None):
        self.name, self.feature, self.n, self.attrs, self.long = name, feature, n, attrs, long
        self.prob, self.prec = prob, prec
        self.plan = plan or {}           # plan facts the GPU test checks (e.g. {"global": 1})
        self.buf, self.sym_offs = build(n, attrs)
        if mutate:
            self.buf = mutate(self.buf)
        self.valid = mutate is None

    def reference(self):
        """Per attribute: (status, symbols) of rans_ref over the attribute's SYMBOLS field, and the buffer's status."""
        res = []
        for a, off in zip(self.attrs, self.sym_offs):
            st, syms, _, _ = R.decode_symbols(self.buf, off, self.n * a.nc, a.nc)
            res.append((st, syms))
        status = next((st for st, _ in res if st != R.OK), R.OK)
        return res, status


def draw(rng, prob, count):
    """`count` symbols, uniform over the table's active entries (narrow ones as often as wide ones)."""
    act = [s for s, p in enumerate(prob) if p]
    return [int(x) for x in rng.choice(act, size=count)]


def table_case(name, feature, prob, prec, rng, n=700, wrap=None, tag=True, long=False, plan=None, final_state=None, pad=0):
    """The three attributes of a table: position (mode 1), int (mode 0) and, when the table is a valid tag table,
    Tagged with this table as its tag table."""
    mbl = MBL[prec]
    syms = draw(rng, prob, 4 * n)
    if wrap is None:
        top = max(s for s, p in enumerate(prob) if p)
        wrap = (-(1 << 20), (1 << 20)) if top > (1 << 20) else (-5, (top + 1) // 2 + 7)
    attrs = [pos_attr(syms[:3 * n], prob, mbl, wrap, final_state, pad), int_attr(syms[3 * n:], prob, mbl, final_state)]
    act = [s for s, p in enumerate(prob) if p]
    if tag and prec == 12 and all(s & 0xFF <= 32 for s in act):
        tags = draw(rng, prob, n)
        vals = [int(rng.integers(0, 1 << (t & 0xFF))) if t & 0xFF else 0 for t in tags for _ in range(2)]
        attrs.append(tag_attr(vals, 2, prob, tags))
    return Case(name, feature, n, attrs, long=long, prob=prob, prec=prec, plan=plan)


# ---- the catalogue ----
def catalogue():
    rng = np.random.default_rng(20261020)
    cases = []
    add = cases.append
    P12, P15 = 1 << 12, 1 << 15

    # degenerate tables
    add(table_case("one_entry", "one entry, prob 2^prec (payload never read)", [P12], 12, rng))
    add(table_case("two_1_rest", "two entries (1, 2^prec-1)", [1, P12 - 1], 12, rng))
    add(table_case("two_rest_1", "two entries (2^prec-1, 1)", [P12 - 1, 1], 12, rng))
    enc = [1, 63, 64, (1 << 14) - 1, 1 << 14, 1 << 18]
    add(table_case("enc_widths", "probabilities in the 1-, 2- and 3-byte encodings", enc + [(1 << 20) - sum(enc)], 20, rng))

    # two-region LUT: first narrow entry at 128m-1, 128m, 128m+1 for kA = 1..7; 2^kA and 2^kA - 1 wide entries, a wide
    # entry behind the narrow run.  The first narrow entry is one slot wide, so it is the first narrow entry for every
    # k <= kA too, and the 2^kA-wide entries in front of it are narrow for every k > kA: kA is the bucket size that
    # needs the fewest LUT bytes (split_choice), the one the device picks
    for ka in range(1, 8):
        for d in (-1, 0, 1):
            s0 = 128 * 4 + d
            w = []
            while s0 - sum(w) >= 2 << ka:
                w.append(1 << ka)
            w.append(s0 - sum(w))
            w += [1] + [max(1, (1 << ka) - 1)] * 64 + [4 << ka]
            prob = table_from_widths(fill(w, P15, 37), gap=2)
            c = table_case("split_ka%d_%+d" % (ka, d), "two-region LUT: first entry narrower than 2^%d at slot %d" % (ka, s0), prob, 15, rng)
            c.expect = {"first_narrow": (ka, s0), "split_k": ka}
            add(c)
    prob = table_from_widths([1] * P12, gap=2)
    c = table_case("split_t0", "two-region LUT with t_split = 0: every entry one slot wide", prob, 12, rng, n=2000, tag=False)
    c.expect = {"first_narrow": (1, 0)}
    add(c)
    prob = table_from_widths(fill([64] * 6 + [1] * 128, P12, 100), gap=2)
    c = table_case("block_128_ones", "a 128-slot block of 128 one-slot entries (block rank 127)", prob, 12, rng, n=1500)
    c.expect = {"first_narrow": (1, 384)}
    add(c)
    prob = table_from_widths(fill([3, 1, 1, 1, 2, 1] * 100, P12, 9), gap=1)
    c = table_case("dense_search", "dense table (uniform LUT only): the probe's search loop runs at every bucket size", prob, 12, rng)
    c.expect = {"dense": True, "search": True}
    add(c)

    # bucket-record tables
    for w in (16, 17):
        prob = table_from_widths(fill([64] * 16 + [3] * 8, P12, w))
        c = table_case("rec_byte_w%d" % w, "bucket records: entries %d slots wide in the byte region" % w, prob, 12, rng)
        c.expect = {"rec": w == 16}
        add(c)
    for ka in range(REC_KA0, REC_KA0 + 4):
        b = 1 << ka
        prob = table_from_widths(fill([b] * (1024 // b) + [2, 16] + [9] * 40 + [3] * 16, P12, 16))
        c = table_case("rec_cuts_ka%d" % ka, "bucket records: three cuts inside the table for kA = %d" % ka, prob, 12, rng)
        c.expect = {"rec_cuts": ka}
        add(c)
    # an entry boundary one slot either side of each cut: the cut moves onto the boundary in front of it (the old cut
    # is then one slot behind it) or stays with a new boundary one slot behind it
    base = table_from_widths(fill([256] * 4 + [2, 16] + [9] * 40 + [3] * 16, P12, 16))
    for i, cut in enumerate(rec_cuts(base, REC_KA0)):
        for d in (-1, 1):
            c = table_case("rec_edge_%s%+d" % ("abc"[i], d), "bucket records: a boundary one slot %s cut t%s" % (
                "in front of" if d < 0 else "behind", "abc"[i]), split_at(base, cut + d), 12, rng)
            c.expect = {"rec_edge": i}
            add(c)
    prob = table_from_widths(fill([64] * 16 + [1] * 40 + [100], P12, 16))
    c = table_case("rec_wide_behind", "bucket records: a wide entry behind narrow ones (no record shape)", prob, 12, rng)
    c.expect = {"rec": False}
    add(c)

    # compact and dense tables, the value map
    for extra, name in ((1, "eq"), (0, "minus1"), (2, "plus1")):
        na = 100
        ns = 2 * na + extra
        prob = random_table(rng, 12, na) + [0] * (ns - na)
        prob = [prob[i] for i in rng.permutation(ns)]
        c = table_case("ns_2na1_%s" % name, "2*n_active+1 vs num_symbols: %d vs %d" % (2 * na + 1, ns), prob, 12, rng, tag=False)
        c.expect = {"compact": 2 * na + 1 < ns}
        add(c)
    base = random_table(rng, 12, 50)
    for where, name in ((0, "0"), (1, "1"), (25, "mid"), (50, "all")):
        prob = base[:where] + [0] + base[where:] + [0] * 200
        c = table_case("dprefix_%s" % name, "compact table, dense prefix of %d" % where, prob, 12, rng, tag=False)
        c.expect = {"dprefix": where, "compact": True}
        add(c)
    prob = table_from_widths(fill([1, 2, 1, 3] * 200, P12, 5), gap=1)
    c = table_case("dense_zero_width", "dense table, zero-width entries between two owners of a bucket", prob, 12, rng)
    c.expect = {"dense": True}
    add(c)
    for ns in (65535, 65536):
        act = sorted(set([0, 1, 2, 777, 4096, 30000] + list(rng.choice(ns - 2, 40, replace=False)) + [ns - 2, ns - 1]))
        w = random_table(rng, 15, len(act))
        prob = [0] * ns
        for s, p in zip(act, w):
            prob[s] = p
        c = table_case("ns_%d" % ns, "num_symbols %d, values %d and %d" % (ns, zz_dec(ns - 2), zz_dec(ns - 1)), prob, 15, rng,
                       wrap=(-40000, 40000))
        c.expect = {"wide": ns > 65535}
        c.plan = {"wide": int(ns > 65535)}
        add(c)

    # precisions
    for prec in (12, 13, 15, 16, 18, 20):
        add(table_case("prec%d" % prec, "precision %d (%s tables)" % (prec, "u16" if prec <= 15 else "u32"),
                       random_table(rng, prec, 300, gap=3), prec, rng))
    add(table_case("table_global", "tables in global memory (lane bytes > 40 KB)", random_table(rng, 20, 20000, gap=2), 20, rng,
                   n=2000, plan={"global": 1}))

    # stream lengths, components, payload lengths and offsets, init tags, final states
    small = random_table(rng, 12, 16)
    for nc in (1, 2, 3, 4):
        for n in (0, 1, 2, 3, 4, 5, 11, 12, 13, 4095, 4097):
            syms = draw(rng, small, n * nc)
            add(Case("len_nc%d_n%d" % (nc, n), "%d entries of %d components" % (n, nc), n,
                     [quant_attr(nc, syms, small, 5, (-3, 20))], long=n > 1000, prob=small, prec=12))
    uni = [256] * 16
    for target in (127, 128, 129, 255, 256, 257):
        for count in range(1, 2000):
            syms = draw(np.random.default_rng(count), uni, count)
            if len(W.rans_payload(syms, uni, 12)) == target:
                break
        else:
            raise AssertionError("no stream with a payload of %d bytes" % target)
        a = int_attr(syms, uni, 5)
        add(Case("payload_%d" % target, "payload of %d bytes (ring: 128)" % target, count, [a], prob=uni, prec=12))
    for pad in range(16):
        syms = draw(rng, uni, 3 * 300)
        c = Case("offset_pad%d" % pad, "payload offset residue mod 16", 300, [pos_attr(syms, uni, 5, (-3, 20), pad=pad)], prob=uni, prec=12)
        add(c)
    two = [1 << 12, 1 << 12]  # precision 13
    for tag, t in ((0, 10), (1, 1000), (2, 1 << 20), (3, (1 << 22) + 1234)):
        fs = final_state_for((4 << 13) + t, 0, two, 13)
        add(Case("init_tag%d" % tag, "init tag %d" % tag, 1, [int_attr([0], two, 9, final_state=fs)], prob=two, prec=13))
    L = 4 << 12
    for fs, name in ((L, "L"), (256 * L - 1, "256L-1"), (77 * L + 12345, "mid")):
        add(table_case("final_%s" % name, "final state %s" % name, small, 12, rng, n=300, final_state=fs))

    # wrap bounds: max_abs_val = md - 1 (lean) and md (not), bounds at +-2^29 and one past
    wt = table_from_widths(fill([], P12, 200))  # ids 0..20: max_abs_val 10
    assert (len(wt) - 1 + 1) >> 1 == 10
    for mn, mx, name in ((0, 10, "md_minus1"), (0, 9, "md"), (-(1 << 29), 1 << 29, "pm2_29"),
                         (-(1 << 29) - 1, 1 << 29, "lo_past"), (-(1 << 29), (1 << 29) + 1, "hi_past")):
        add(table_case("wrap_%s" % name, "wrap bounds [%d, %d], max |correction| 10" % (mn, mx), wt, 12, rng, wrap=(mn, mx)))
    return cases


def malformed():
    """Buffers the reference decodes to a failure or to symbols other than the encoded ones."""
    rng = np.random.default_rng(7)
    cases = []
    small = random_table(rng, 12, 16)
    n = 3000
    syms = draw(rng, small, 3 * n)
    field = W.symbols_raw_table(syms, small, 5)
    pay = W.rans_payload(syms, small, 12)
    head = field[:len(field) - len(pay) - len(W.varint(len(pay)))]
    for cut in (len(pay) // 2, 40, 3, 2, 1):  # the payload loses its first bytes: the decode runs out before its end
        f = head + W.varint(len(pay) - cut) + pay[cut:]
        cases.append(Case("cut_pos_%d" % cut, "payload short by %d bytes" % cut, n, [pos_attr(syms, small, 5, (-3, 20), field=f)],
                          prob=small, prec=12))

    def raw_field(prob, mbl, pay):
        return bytes([1, mbl]) + W.table_bytes(prob) + W.varint(len(pay)) + pay

    ok_pay = W.rans_payload([0, 1, 2], [1024] * 4, 12)
    bad = [("sum_low", [1024] * 3 + [1023], ok_pay), ("sum_high", [1024] * 3 + [1025], ok_pay),
           ("overflow", [(1 << 22) - 1] * 3, ok_pay), ("init_tag_long", [1024] * 4, bytes([0xC0])),
           ("init_tag_long2", [1024] * 4, bytes([0x12, 0x80])), ("x_ge_256L", [1024] * 4, bytes([0xFF, 0xFF, 0xBF])),
           ("empty_payload", [1024] * 4, b""), ("zero_symbols", [], ok_pay)]
    for name, prob, p in bad:
        cases.append(Case("bad_" + name, "malformed: " + name, 1, [int_attr([0], None, 5, field=raw_field(prob, 5, p))]))

    # Tagged: hand-made tag tables, ids >= 256 cast to a byte, tag 0, tag 33, bit areas at / one bit beyond the end
    tprob = [0] * 33
    for t, p in ((0, 500), (1, 300), (5, 1000), (8, 700), (16, 900), (31, 296), (32, 400)):
        tprob[t] = p
    hi = [0] * 300
    for t, p in ((256 + 3, 2000), (256 + 32, 1000), (256, 500), (7, 596)):
        hi[t] = p
    t33 = list(tprob)
    t33[33 - 1] -= 1
    t33 += [1]
    for name, prob, ntag, want33 in (("hand", tprob, 0, False), ("ids_ge_256", hi, 0, False), ("tag33", t33, 0, True)):
        tags = draw(rng, prob, 400)
        if want33:
            tags[250] = 33
        elif name == "hand":
            tags[:3] = [0, 32, 0]
        vals = [int(rng.integers(0, 1 << (t & 0xFF))) if t & 0xFF else 0 for t in tags for _ in range(3)]
        field = W.symbols_tagged_table(vals, 3, prob, tags)
        cases.append(Case("tags_" + name, "Tagged: " + name, 400, [tag_attr(vals, 3, prob, tags, field=field)], prob=prob, prec=12))
    # bit area exactly at the buffer end (8k bits) and one bit beyond it (8k + 1 bits, last byte cut)
    for name, widths in (("end_exact", [5, 3, 8]), ("one_bit_beyond", [5, 3, 8, 1])):
        tp = [0] * 9
        for t in set(widths):
            tp[t] = 1
        tp[8] += (1 << 12) - sum(tp)
        vals = [int(rng.integers(0, 1 << w)) for w in widths]
        a = tag_attr(vals, 1, tp, widths)
        _, bits = W.tagged_bits(vals, 1, widths)
        cut = (lambda b: b[:-1]) if bits % 8 else None
        cases.append(Case("tags_" + name, "Tagged: bit area of %d bits, buffer ends at bit %d" % (bits, bits // 8 * 8), len(widths),
                          [a], mutate=cut, prob=tp, prec=12))
    # the payload of a tag stream cut short: the tag loop runs out of bytes
    tags = draw(rng, tprob, 3000)
    vals = [int(rng.integers(0, 1 << (t & 0xFF))) if t & 0xFF else 0 for t in tags]
    full = W.symbols_tagged_table(vals, 1, tprob, tags)
    tpay = W.rans_payload(tags, tprob, 12)
    hdr = bytes([0]) + W.table_bytes(tprob)
    bits = full[len(hdr) + len(W.varint(len(tpay))) + len(tpay):]
    for cut in (len(tpay) // 2, 2):
        f = hdr + W.varint(len(tpay) - cut) + tpay[cut:] + bits
        cases.append(Case("tags_cut_%d" % cut, "Tagged: tag payload short by %d bytes" % cut, 3000, [tag_attr(vals, 1, tprob, tags, field=f)],
                          prob=tprob, prec=12))
    for c in cases:
        c.valid = False
    return cases


def rec_limit(num_sms, ka):
    """The record-kernel tables nearest the planner's shared-memory limit for wide-region buckets of 2^ka slots: a
    dense precision-15 table whose byte region starts at slot T (a wide region of 256-slot entries in front of it).
    16 * num_sms streams give every SM 16 streams: 4 warp pairs of 4 lanes.  Returns (accepted, refused): the cases
    of the smallest T whose tables the planner still accepts and of the next smaller one, each with .rec_bytes."""
    P, lanes, pairs, ksym = 1 << 15, 4, 4, 12
    rng = np.random.default_rng(ka)

    def table(T):
        w = [256] * (T // 256) + ([T % 256] if T % 256 else []) + [3, 3, 3]
        return table_from_widths(fill(w, P, 16))

    def fits(T):
        return rec_fits(lanes, pairs, rec_bytes(table(T), ka), ksym)

    lo, hi = 8, P - 1024  # lo: refused, hi: accepted
    assert not fits(lo) and fits(hi)
    while hi - lo > 8:
        mid = (lo + hi) // 2 & ~7
        lo, hi = (lo, mid) if fits(mid) else (mid, hi)
    out = []
    for T in (hi, lo):
        prob = table(T)
        syms = draw(rng, prob, 3 * 64)
        c = Case("rec_limit_ka%d_T%d" % (ka, T), "record tables at the planner's limit, byte region from slot %d" % T, 64,
                 [pos_attr(syms, prob, MBL[15], (-5, 1000))], prob=prob, prec=15)
        c.rec_bytes = rec_bytes(prob, ka)
        c.n_bufs = 16 * num_sms
        out.append(c)
    return out


def no_split(num_sms):
    """A compact precision-15 table whose first entry is one slot wide: for every kA the two-region LUT's narrow
    region would cover all 2^15 slots (16 KB per lane).  8 * num_sms streams leave each lane less than that, so the
    device finds no feasible split and probes the uniform LUT, whose buckets meet several entries."""
    rng = np.random.default_rng(8)
    prob = table_from_widths([1] + [4] * ((1 << 15) // 4 - 1) + [3], gap=2)
    syms = draw(rng, prob, 3 * 100)
    c = Case("no_split", "compact table without a feasible split", 100, [pos_attr(syms, prob, MBL[15], (-5, 30000))],
             prob=prob, prec=15)
    c.n_bufs = 8 * num_sms
    return c


def warp_mix(num_sms):
    """31 lean-eligible streams and one that is not (its largest correction reaches max_diff) in the first warp of one
    group: all have the same table, length and group key; the rest of the batch fills the machine so that the group
    runs 32 lanes per warp.  Returns (buffers, index of the odd one, the two cases)."""
    rng = np.random.default_rng(32)
    wt = table_from_widths(fill([], 1 << 12, 200))
    syms = draw(rng, wt, 3 * 64)
    lean = Case("mix_lean", "lean", 64, [pos_attr(syms, wt, 5, (0, 10))])
    odd = Case("mix_odd", "not lean", 64, [pos_attr(syms, wt, 5, (0, 9))])
    bufs = [lean.buf] * (num_sms * 128)
    bufs[5] = odd.buf
    return bufs, 5, lean, odd
