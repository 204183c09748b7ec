"""Minimal pure-Python Draco v2.2 bitstream writer for tests (point clouds, sequential attribute encoding).

Independent of the C++ generator (draco_sharp_b200/synth): it lets a test choose the *corrections* directly,
so it can build streams no real encoder would (irregular wrap corrections, uncompressed integers, generic
attributes, degenerate alphabets, every max_bit_length) and corrupt ones.  Layout per SURVEY.md Appendix A.
"""
import struct

import numpy as np


def varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        if v:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def rans_precision(mbl):
    return min(20, max(12, (3 * mbl) // 2))


def zigzag(v):
    v = int(v)
    return (v << 1) if v >= 0 else (((-(v + 1)) << 1) | 1)


def normalize_probs(freq, prec_bits):
    """Integer probabilities summing to 2^prec_bits, >= 1 for every symbol that occurs."""
    P = 1 << prec_bits
    freq = np.asarray(freq, dtype=np.int64)
    total = int(freq.sum())
    prob = np.zeros(len(freq), dtype=np.int64)
    nz = freq > 0
    prob[nz] = np.maximum(1, (freq[nz] * P) // total)
    diff = P - int(prob.sum())
    order = np.argsort(-prob)
    i = 0
    while diff != 0:
        j = order[i % len(order)]
        if diff > 0:
            prob[j] += diff
            diff = 0
        elif prob[j] > 1:
            take = min(prob[j] - 1, -diff)
            prob[j] -= take
            diff += take
        i += 1
    assert prob.sum() == P and (prob[nz] >= 1).all()
    return prob


def table_bytes(prob, pad=0):
    """RANS_TABLE.  pad: write that many extra bytes by giving the first non-zero probabilities a longer encoding than
    they need (a zero extra byte); the decoder reads the same table, the payload behind it moves by `pad` bytes."""
    out = bytearray(varint(len(prob)))
    i = 0
    n = len(prob)
    while i < n:
        p = int(prob[i])
        if p == 0:
            off = 0
            while off < 63 and i + off + 1 < n and prob[i + off + 1] == 0:
                off += 1
            out.append((off << 2) | 3)
            i += off + 1
        else:
            extra = 0 if p < (1 << 6) else (1 if p < (1 << 14) else 2)
            more = min(pad, 2 - extra)
            extra += more
            pad -= more
            out.append(((p << 2) & 0xFC) | extra)
            for b in range(extra):
                out.append((p >> (8 * (b + 1) - 2)) & 0xFF)
            i += 1
    assert pad == 0, "not enough entries to pad the table"
    return bytes(out)


def rans_payload(symbols, prob, prec_bits, final_state=None):
    """rANS payload of `symbols` under `prob`.  final_state: the state the decoder ends in (the encoder's initial
    state, in [L, 256 L)); L by default."""
    P = 1 << prec_bits
    l_base = 4 * P
    cum = np.concatenate([[0], np.cumsum(prob)])
    state = l_base if final_state is None else int(final_state)
    assert l_base <= state < 256 * l_base
    buf = bytearray()
    for s in reversed([int(x) for x in symbols]):
        p = int(prob[s])
        lim = (l_base // P) * 256 * p
        while state >= lim:
            buf.append(state & 0xFF)
            state >>= 8
        state = (state // p) * P + state % p + int(cum[s])
    s = state - l_base
    if s < (1 << 6):
        buf.append(s)
    elif s < (1 << 14):
        v = (1 << 14) + s
        buf += bytes([v & 0xFF, v >> 8])
    elif s < (1 << 22):
        v = (2 << 22) + s
        buf += bytes([v & 0xFF, (v >> 8) & 0xFF, v >> 16])
    else:
        v = (3 << 30) + s
        buf += bytes([v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF, v >> 24])
    return bytes(buf)


def symbols_raw(symbols, mbl=None):
    """SYMBOLS field, Raw scheme (scheme byte 1)."""
    symbols = [int(s) for s in symbols]
    if not symbols:
        return b""
    freq = np.bincount(np.asarray(symbols, dtype=np.int64))
    if mbl is None:
        nu = int((freq > 0).sum())
        mbl = min(18, max(1, nu.bit_length()))
    pb = rans_precision(mbl)
    prob = normalize_probs(freq, pb)
    pay = rans_payload(symbols, prob, pb)
    return bytes([1, mbl]) + table_bytes(prob) + varint(len(pay)) + pay


def _check_table(prob, prec_bits, symbols):
    prob = [int(p) for p in prob]
    assert sum(prob) == 1 << prec_bits, "probabilities must sum to 2^%d" % prec_bits
    assert all(0 <= s < len(prob) and prob[s] > 0 for s in symbols), "a symbol without probability"
    return prob


def symbols_raw_table(symbols, prob, mbl, final_state=None, pad=0):
    """SYMBOLS field, Raw scheme, with a probability table the caller chooses (not derived from the symbols): any
    table summing to 2^precision(mbl), symbols with a probability that never occur included."""
    symbols = [int(s) for s in symbols]
    if not symbols:
        return b""
    pb = rans_precision(mbl)
    prob = _check_table(prob, pb, symbols)
    pay = rans_payload(symbols, prob, pb, final_state)
    return bytes([1, mbl]) + table_bytes(prob, pad) + varint(len(pay)) + pay


def tagged_bits(symbols, nc, tags):
    """The LSB-first bit area of a Tagged stream: per point, nc fields of (tags[i] & 0xFF) bits.  Returns (bytes, bits)."""
    acc, nacc, bits, total = 0, 0, bytearray(), 0
    for i, t in enumerate(tags):
        w = int(t) & 0xFF
        for c in range(nc):
            acc |= (int(symbols[i * nc + c]) & ((1 << w) - 1)) << nacc
            nacc += w
            total += w
            while nacc >= 8:
                bits.append(acc & 0xFF)
                acc >>= 8
                nacc -= 8
    if nacc:
        bits.append(acc & 0xFF)
    return bytes(bits), total


def symbols_tagged_table(symbols, nc, tag_prob, tags=None, final_state=None):
    """SYMBOLS field, Tagged scheme, with a tag table the caller chooses (precision 12).  tags: the tag symbol of every
    point (default: the bit length of its largest value); the decoder uses tag & 0xFF as the field width."""
    symbols = [int(s) for s in symbols]
    if not symbols:
        return b""
    n = len(symbols) // nc
    if tags is None:
        tags = [max(1, max(symbols[i * nc:(i + 1) * nc]).bit_length()) for i in range(n)]
    tags = [int(t) for t in tags]
    tag_prob = _check_table(tag_prob, 12, tags)
    pay = rans_payload(tags, tag_prob, 12, final_state)
    return bytes([0]) + table_bytes(tag_prob) + varint(len(pay)) + pay + tagged_bits(symbols, nc, tags)[0]


def symbols_tagged(symbols, nc):
    """SYMBOLS field, Tagged scheme (scheme byte 0): one bit-length tag per point, LSB-first bit fields."""
    symbols = [int(s) for s in symbols]
    if not symbols:
        return b""
    n = len(symbols) // nc
    tags = []
    for i in range(n):
        m = max(symbols[i * nc:(i + 1) * nc])
        tags.append(max(1, m.bit_length()))
    freq = np.bincount(np.asarray(tags, dtype=np.int64), minlength=1)
    prob = normalize_probs(freq, 12)
    pay = rans_payload(tags, prob, 12)
    acc = 0
    nacc = 0
    bits = bytearray()
    for i in range(n):
        for c in range(nc):
            acc |= (symbols[i * nc + c] & ((1 << tags[i]) - 1)) << nacc
            nacc += tags[i]
            while nacc >= 8:
                bits.append(acc & 0xFF)
                acc >>= 8
                nacc -= 8
    if nacc:
        bits.append(acc & 0xFF)
    return bytes([0]) + table_bytes(prob) + varint(len(pay)) + pay + bytes(bits)


def portable_int(corr, nc, pred_method=0, transform=1, scheme="raw", pred_data=b"", zig=True, num_bytes=None, mbl=None,
                 prob=None, tag_prob=None, tags=None):
    """PORTABLE(int-like): corrections (flat, entry-major) -> bytes.  prob (Raw, with mbl) / tag_prob (Tagged, with
    optional tags): a caller-chosen table instead of one derived from the symbols."""
    out = bytearray(struct.pack("<b", pred_method))
    if pred_method != -2:
        out += struct.pack("<b", transform)
    syms = [zigzag(c) if zig else int(c) for c in corr]
    if scheme == "uncompressed":
        out.append(0)
        out.append(num_bytes)
        for s in syms:
            out += int(s & ((1 << (8 * num_bytes)) - 1)).to_bytes(num_bytes, "little") if num_bytes else b""
    else:
        out.append(1)
        if scheme == "raw":
            out += symbols_raw(syms, mbl) if prob is None else symbols_raw_table(syms, prob, mbl)
        else:
            out += symbols_tagged(syms, nc) if tag_prob is None else symbols_tagged_table(syms, nc, tag_prob, tags)
    out += pred_data
    return bytes(out)


def rabs_block(bits, prob_zero=None):
    """A bit sequence as RAnsBitEncoder leaves it (Draco ans.h rabs_desc_write / ans_write_end): u8 prob_zero | varint
    size | rABS bytes.  A RAnsBitDecoder reads the bits back in the order given (BitCoders/RAnsBitDecoder.cs:12-35)."""
    bits = [1 if b else 0 for b in bits]
    if prob_zero is None:
        zeros = len(bits) - sum(bits)
        prob_zero = min(255, max(1, int(256.0 * zeros / max(1, len(bits)) + 0.5)))
    p0, p1 = prob_zero, 256 - prob_zero
    state, data = 4096, bytearray()
    for b in reversed(bits):
        ls = p1 if b else p0
        if state >= 4096 * ls:
            data.append(state & 0xFF)
            state >>= 8
        quot, rem = divmod(state, ls)
        state = quot * 256 + rem + (0 if b else p1)
    state -= 4096
    if state < (1 << 6):
        data.append(state)
    elif state < (1 << 14):
        data += int((1 << 14) + state).to_bytes(2, "little")
    else:
        assert state < (1 << 22)
        data += int((2 << 22) + state).to_bytes(3, "little")
    return bytes([prob_zero]) + varint(len(data)) + bytes(data)


def tex_coords_data(flags, mn, mx, prob_zero=None):
    """PRED_DATA of MeshPredictionSchemeTexCoordsPortableDecoder (:68-84): i32 count, rABS flags where a 0 bit FLIPS the
    running orientation (starting from true), then the wrap transform's bounds."""
    bits, last = [], True
    for f in flags:
        bits.append(1 if bool(f) == last else 0)
        last = bool(f)
    return struct.pack("<i", len(bits)) + rabs_block(bits, prob_zero) + wrap_data(mn, mx)


def cmp_data(crease, mn, mx):
    """PRED_DATA of MeshPredictionSchemeConstrainedMultiParallelogramDecoder (DecodeTransformData :119-141, v2.2: no mode
    byte): per context (1..4 parallelograms) a varint flag count and, when it is not zero, the rABS-coded crease flags;
    then the wrap transform's bounds."""
    out = bytearray()
    for ctx in range(4):
        bits = list(crease[ctx]) if ctx < len(crease) else []
        out += varint(len(bits))
        if bits:
            out += rabs_block(bits)
    return bytes(out) + wrap_data(mn, mx)


def cmp_encode(values, nc, maps, mn, mx, rng, p_crease=0.3, max_par=4):
    """Encoder side of the constrained multi-parallelogram scheme, written from the Draco bitstream specification
    (independent of oracle/ and of the CUDA path): for every entry, the parallelograms found swinging left then right
    around its corner, random crease flags, the truncated mean of the kept predictions, and the wrapped correction.
    Returns (corrections, [flags of context 0..3])."""
    INV = 0xFFFFFFFF
    opp, c2v = maps["opposite"], maps["corner_to_vertex"]
    d2c, v2d = maps["data_to_corner"], maps["vertex_to_data"]
    n = len(values) // nc
    vals = [int(v) for v in values]
    nxt = lambda c: INV if c == INV else (c - 2 if c % 3 == 2 else c + 1)
    prv = lambda c: INV if c == INV else (c + 2 if c % 3 == 0 else c - 1)
    op = lambda c: INV if c == INV else int(opp[c])
    max_diff = 1 + mx - mn
    max_corr = max_diff // 2
    min_corr = -max_corr
    if max_diff % 2 == 0:
        max_corr -= 1
    trunc_div = lambda a, b: abs(a) // b * (1 if a >= 0 else -1)
    to_i32 = lambda v: ((v + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)
    corr, crease = [], [[], [], [], []]

    def emit(p, pred):
        for c in range(nc):
            q = min(max(pred[c], mn), mx)
            d = vals[p * nc + c] - q
            if d < min_corr:
                d += max_diff
            elif d > max_corr:
                d -= max_diff
            corr.append(d)

    emit(0, [0] * nc)
    for p in range(1, n):
        start = int(d2c[p])
        corner, first, found = start, True, []
        while corner != INV:
            oc = op(corner)
            if oc != INV:
                e = [int(v2d[int(c2v[x])]) for x in (oc, nxt(oc), prv(oc))]
                if all(x < p for x in e):
                    found.append(e)
                    if len(found) == max_par:
                        break
            corner = nxt(op(nxt(corner))) if first else prv(op(prv(corner)))
            if corner == start:
                break
            if corner == INV and first:
                first = False
                corner = prv(op(prv(start)))
        kept = []
        for e in found:
            f = bool(rng.random() < p_crease)
            crease[len(found) - 1].append(1 if f else 0)
            if not f:
                kept.append(e)
        if not kept:
            emit(p, vals[(p - 1) * nc: p * nc])
        else:
            pred = []
            for c in range(nc):
                sm = 0
                for (eo, en, ep) in kept:
                    sm = to_i32(sm + to_i32(vals[en * nc + c] + vals[ep * nc + c] - vals[eo * nc + c]))
                pred.append(trunc_div(sm, len(kept)))
            emit(p, pred)
    return corr, crease


def geometric_normal_data(flips, bits, canonical=True):
    """PRED_DATA of MeshPredictionSchemeGeometricNormalDecoder (DecodePredictionData :72-82, v2.2: no mode byte): the
    octahedron transform's data (i32 max_quantized_value [, i32 center_value]) and then the rABS-coded flip bits."""
    max_q = (1 << bits) - 1
    out = struct.pack("<i", max_q)
    if canonical:
        out += struct.pack("<i", (max_q - 1) // 2)
    return out + rabs_block(flips)


def geometric_normal_predictions(maps, pos_maps, pos_values, bits, flips):
    """Predicted octahedral coordinates of every entry under the geometric-normal scheme, written from the Draco bitstream
    specification (independent of oracle/ and of the CUDA path): area-weighted normal of the triangles around the
    entry's vertex in position space, scaled below 2^29, canonicalised to an L1 norm of the centre value, flipped, then
    mapped to canonical octahedral coordinates.  Python integers emulate the int64 / int32 wrapping."""
    INV = 0xFFFFFFFF
    opp, d2c = maps["opposite"], maps["data_to_corner"]
    p_c2v, p_v2d = pos_maps["corner_to_vertex"], pos_maps["vertex_to_data"]
    nxt = lambda c: INV if c == INV else (c - 2 if c % 3 == 2 else c + 1)
    prv = lambda c: INV if c == INV else (c + 2 if c % 3 == 0 else c - 1)
    op = lambda c: INV if c == INV else int(opp[c])
    wrap64 = lambda v: ((v + (1 << 63)) & ((1 << 64) - 1)) - (1 << 63)
    wrap32 = lambda v: ((v + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)
    tdiv = lambda a, b: abs(a) // abs(b) * (1 if (a >= 0) == (b >= 0) else -1)
    max_q = (1 << bits) - 1
    max_value = max_q - 1
    center = max_value // 2

    def pos_of(c):
        e = int(p_v2d[int(p_c2v[c])])
        return [int(x) for x in pos_values[3 * e: 3 * e + 3]]

    preds = []
    for p in range(len(d2c)):
        start = int(d2c[p])
        cent = pos_of(start)
        corners, c = [], start
        while c != INV:                      # all corners around the vertex: swing left, then right from the start
            corners.append(c)
            c = nxt(op(nxt(c)))
            if c == start:
                c = INV
        if nxt(op(nxt(corners[-1]))) == INV:  # open fan: continue on the right-hand side
            c = prv(op(prv(start)))
            while c != INV:
                corners.append(c)
                c = prv(op(prv(c)))
        nrm = [0, 0, 0]
        for c in corners:
            a = [x - y for x, y in zip(pos_of(nxt(c)), cent)]
            b = [x - y for x, y in zip(pos_of(prv(c)), cent)]
            cr = [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]
            nrm = [wrap64(x + y) for x, y in zip(nrm, cr)]
        abs_sum = min(sum(abs(x) for x in nrm), (1 << 63) - 1)
        if abs_sum > (1 << 29):
            q = abs_sum // (1 << 29)
            nrm = [tdiv(x, q) for x in nrm]
        v = [wrap32(x) for x in nrm]
        l1 = abs(v[0]) + abs(v[1]) + abs(v[2])
        if l1 == 0:
            v[0] = center
        else:
            v[0] = tdiv(v[0] * center, l1)
            v[1] = tdiv(v[1] * center, l1)
            rest = center - abs(v[0]) - abs(v[1])
            v[2] = rest if v[2] >= 0 else -rest
        if flips[p]:
            v = [-x for x in v]
        if v[0] >= 0:
            s_, t_ = v[1] + center, v[2] + center
        else:
            s_ = abs(v[2]) if v[1] < 0 else max_value - abs(v[2])
            t_ = abs(v[1]) if v[2] < 0 else max_value - abs(v[1])
        if (s_, t_) in ((0, 0), (0, max_value), (max_value, 0)):
            s_, t_ = max_value, max_value
        elif s_ == 0 and t_ > center:
            t_ = center - (t_ - center)
        elif s_ == max_value and t_ < center:
            t_ = center + (center - t_)
        elif t_ == max_value and s_ < center:
            s_ = center + (center - s_)
        elif t_ == 0 and s_ > center:
            s_ = center - (s_ - center)
        preds += [s_, t_]
    return preds


def wrap_data(mn, mx):
    return struct.pack("<ii", mn, mx)


def quant_params(mins, rng, bits):
    return b"".join(struct.pack("<f", m) for m in mins) + struct.pack("<f", rng) + bytes([bits])


def point_cloud(n_points, attrs, version=(2, 2), geom_type=0, method=0, flags=0, decoders=None):
    """attrs: list of dicts {att_type, data_type, nc, normalized, unique_id, seq_type, portable, xform}.
    decoders: list of lists of attribute indices (default: one decoder with all attributes)."""
    out = bytearray(b"DRACO" + bytes([version[0], version[1], geom_type, method]) + struct.pack("<H", flags))
    out += struct.pack("<i", n_points)
    if decoders is None:
        decoders = [list(range(len(attrs)))]
    out.append(len(decoders))
    for dec in decoders:
        out += varint(len(dec))
        for i in dec:
            a = attrs[i]
            out += bytes([a["att_type"], a["data_type"], a["nc"], a.get("normalized", 0)]) + varint(a.get("unique_id", i))
        for i in dec:
            out.append(attrs[i]["seq_type"])
    for dec in decoders:
        for i in dec:
            out += attrs[i]["portable"]
        for i in dec:
            out += attrs[i].get("xform", b"")
    return bytes(out)


def sequential_mesh(faces, n_points, attrs, method=0, scheme="raw", decoders=None):
    """A v2.2 sequential mesh (MeshSequentialDecoder.cs:8-118): header, varint faces / points, u8 method, indices
    (method 0: index differences as symbols, magnitude << 1 with bit 0 set for negative ones; method 1: plain indices,
    width by point count), then the ATTRIBUTES section of point_cloud()."""
    faces = [int(v) for f in faces for v in f]
    out = bytearray(b"DRACO" + bytes([2, 2, 1, 0]) + struct.pack("<H", 0))
    out += varint(len(faces) // 3) + varint(n_points)
    out.append(method)
    if method == 0:
        syms, last = [], 0
        for v in faces:
            d = v - last
            syms.append((abs(d) << 1) | (1 if d < 0 else 0))
            last = v
        if syms:
            out += symbols_raw(syms) if scheme == "raw" else symbols_tagged(syms, 1)
    else:
        for v in faces:
            if n_points < 256:
                out.append(v)
            elif n_points < (1 << 16):
                out += struct.pack("<H", v)
            elif n_points < (1 << 21):
                out += varint(v)
            else:
                out += struct.pack("<I", v)
    body = point_cloud(n_points, attrs, decoders=decoders)
    return bytes(out) + body[15:]  # point_cloud(): 11-byte header + int32 point count, then the ATTRIBUTES section
