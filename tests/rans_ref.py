"""Plain restatement of the reference's symbol decoding, with Python integers.  TEST INFRASTRUCTURE.

RAnsSymbolDecoder.Create / StartDecoding (Entropy/RAnsSymbolDecoder.cs:12-59), RAnsDecoder.ReadInit / Read /
BuildLookupTable (Entropy/RAnsDecoder.cs:20-99) and SymbolDecoding.DecodeSymbols (Entropy/SymbolDecoding.cs:7-67),
with the Tagged bit fields read LSB-first into a full 32-bit value (SURVEY.md Appendix B-3 / B-4).  It exists for
malformed streams, where the expected output is what the reference decodes rather than the symbols that were encoded.
Statuses are the C ABI's DCB_ERR_* numbers.
"""

OK, EOF, SCHEME, BITLEN, TABLE, RANS_INIT, TAG, NUM_SYMBOLS = 0, -1, -4, -5, -6, -7, -12, -13


class Fail(Exception):
    def __init__(self, status):
        self.status = status


class Reader:
    def __init__(self, buf, pos=0):
        self.buf, self.pos = bytes(buf), pos

    def u8(self):
        if self.pos >= len(self.buf):
            raise Fail(EOF)
        self.pos += 1
        return self.buf[self.pos - 1]

    def varint(self):  # DecoderBuffer.cs:26-42
        v = 0
        for i in range(10):
            b = self.u8()
            v |= (b & 0x7F) << (7 * i)
            if not b & 0x80:
                return v
        raise Fail(EOF)


def precision(mbl):  # RAnsSymbolCoding.cs:10-26
    return min(20, max(12, (3 * mbl) // 2))


class RAns:
    def __init__(self, rd, mbl):
        """RAnsSymbolDecoder.Create (:12-51) + BuildLookupTable (RAnsDecoder.cs:69-88)."""
        self.prec_bits = precision(mbl)
        self.P = 1 << self.prec_bits
        self.L = 4 * self.P
        ns = rd.varint()
        self.prob = [0] * ns
        i = 0
        while i < ns:
            pd = rd.u8()
            if pd & 3 == 3:
                if i + (pd >> 2) >= ns:
                    raise Fail(TABLE)  # :31
                i += (pd >> 2) + 1
                continue
            p = pd >> 2
            for b in range(pd & 3):
                p |= rd.u8() << (8 * (b + 1) - 2)
            self.prob[i] = p
            i += 1
        self.cum, c = [], 0
        for p in self.prob:
            self.cum.append(c)
            c += p
            if c > self.P:
                raise Fail(TABLE)  # RAnsDecoder.cs:80
        if ns and c != self.P:
            raise Fail(TABLE)  # :87
        self.lut = [0] * self.P
        for s, (p, c0) in enumerate(zip(self.prob, self.cum)):
            self.lut[c0:c0 + p] = [s] * p

    def start(self, rd):
        """StartDecoding (:53-59) + ReadInit (RAnsDecoder.cs:20-54)."""
        n = rd.varint()
        if rd.pos + n > len(rd.buf):
            raise Fail(EOF)
        self.data = rd.buf[rd.pos:rd.pos + n]
        rd.pos += n
        if n < 1:
            raise Fail(RANS_INIT)
        tag = self.data[n - 1] >> 6
        if n < tag + 1:
            raise Fail(RANS_INIT)
        self.off = n - (tag + 1)
        x = int.from_bytes(self.data[self.off:n], "little") & ((1 << (8 * tag + 6)) - 1)
        self.state = x + self.L
        if self.state >= self.L * 256:
            raise Fail(RANS_INIT)  # :53

    def read(self):
        """Read (:56-67) + FetchSymbol (:90-99)."""
        while self.state < self.L and self.off > 0:
            self.off -= 1
            self.state = self.state * 256 + self.data[self.off]
        q, r = self.state >> self.prec_bits, self.state & (self.P - 1)
        s = self.lut[r]
        self.state = q * self.prob[s] + r - self.cum[s]
        return s


def decode_symbols(buf, pos, num_values, nc):
    """SymbolDecoding.DecodeSymbols over buf[pos:] (buf runs to the end of the .drc buffer: the Tagged bit area has no
    length of its own).  Returns (status, symbols, end position, final rANS state); symbols decoded before a failure
    are kept."""
    out = []
    if num_values == 0:
        return OK, out, pos, None  # :9-13
    rd = Reader(buf, pos)
    a = None
    try:
        scheme = rd.u8()
        if scheme == 0:  # Tagged :30-50
            a = RAns(rd, 5)
            if not a.prob:
                raise Fail(NUM_SYMBOLS)  # :36
            a.start(rd)
            bit0 = bitpos = rd.pos * 8
            while len(out) < num_values:
                width = a.read() & 0xFF  # (byte) cast :41
                if width > 32:
                    raise Fail(TAG)  # DecoderBuffer.cs:141
                for _ in range(nc):
                    if len(out) == num_values:
                        break
                    if bitpos + width > 8 * len(rd.buf):
                        raise Fail(EOF)
                    v = int.from_bytes(rd.buf[bitpos >> 3:(bitpos + width + 7) // 8 + 1], "little")
                    out.append((v >> (bitpos & 7)) & ((1 << width) - 1))
                    bitpos += width
            rd.pos += (bitpos - bit0 + 7) // 8  # EndBitDecoding: ceil(bits / 8) (B-4)
        elif scheme == 1:  # Raw :52-67
            mbl = rd.u8()
            if mbl < 1 or mbl > 18:
                raise Fail(BITLEN)  # :56
            a = RAns(rd, mbl)
            if not a.prob:
                raise Fail(NUM_SYMBOLS)  # :59
            a.start(rd)
            out = [a.read() for _ in range(num_values)]
        else:
            raise Fail(SCHEME)  # :26
    except Fail as f:
        return f.status, out, rd.pos, None
    return OK, out, rd.pos, a.state
