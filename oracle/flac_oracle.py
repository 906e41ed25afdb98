"""FLAC (RFC 9639) test infrastructure: a NumPy encoder that can force every coding choice, and a plain Python decoder.

Neither is used by the package.  The encoder writes streams whose every feature is chosen by the test (subframe type
and order, LPC precision and shift, Rice method and partition order, escaped partitions, wasted bits, stereo mode,
fixed or variable blocking, block sizes, header codes, metadata blocks); the decoder is the independent statement of
the grammar the device decoder is checked against.
"""
import numpy as np

STEREO = {"independent": 1, "left_side": 8, "side_right": 9, "mid_side": 10}
RATE_CODES = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10,
              96000: 11}
SIZE_CODES = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6, 32: 7}


def crc8(data, crc=0):
    for b in data:
        crc ^= b
        for _ in range(8):
            crc = ((crc << 1) ^ 0x07) & 0xFF if crc & 0x80 else (crc << 1) & 0xFF
    return crc


_CRC16 = []
for _b in range(256):
    _c = _b << 8
    for _ in range(8):
        _c = ((_c << 1) ^ 0x8005) & 0xFFFF if _c & 0x8000 else (_c << 1) & 0xFFFF
    _CRC16.append(_c)


def crc16(data, crc=0):
    tab = _CRC16
    for b in data:
        crc = ((crc << 8) & 0xFFFF) ^ tab[(crc >> 8) ^ b]
    return crc


def utf8_number(v):
    """FLAC's UTF-8-style coded number (up to 36 bits)."""
    if v < 0x80:
        return bytes([v])
    for n in range(2, 8):                      # total bytes
        if v < (1 << (5 * n + 1)) or n == 7:
            break
    out = []
    for _ in range(n - 1):
        out.append(0x80 | (v & 0x3F))
        v >>= 6
    lead = (0xFF << (8 - n)) & 0xFF
    out.append(lead | v)
    return bytes(reversed(out))


class Sub:
    """Coding of one subframe.  kind: "constant" | "verbatim" | "fixed" | "lpc"; order: predictor order;
    precision / shift: LPC coefficient precision and shift (None: 12 / chosen from the coefficients); method: 0
    (4-bit Rice parameters) or 1 (5-bit); porder: partition order (None: the largest that divides the block, up to
    4); escape: partition indices sent as raw signed values; escape_width: their width (None: the smallest that
    holds them); wasted: wasted bits k (every sample must be a multiple of 2^k)."""

    def __init__(self, kind="fixed", order=2, precision=None, shift=None, method=0, porder=None, escape=(),
                 escape_width=None, wasted=0, rice=None):
        self.kind, self.order, self.precision, self.shift = kind, order, precision, shift
        self.method, self.porder, self.escape, self.escape_width = method, porder, tuple(escape), escape_width
        self.wasted, self.rice = wasted, rice


def _fields_to_bits(vals, nbits):
    """Big-endian bit array (uint8 0/1) of fields (value, width); a width above 64 is leading zeros."""
    vals = np.asarray(vals, dtype=np.uint64)
    nbits = np.asarray(nbits, dtype=np.int64)
    keep = nbits > 0
    vals, nbits = vals[keep], nbits[keep]
    if nbits.size == 0:
        return np.zeros(0, np.uint8)
    starts = np.cumsum(nbits) - nbits
    fid = np.repeat(np.arange(nbits.size), nbits)
    j = np.arange(int(nbits.sum())) - starts[fid]
    sh = nbits[fid] - 1 - j
    bit = (vals[fid] >> np.minimum(sh, 63).astype(np.uint64)) & np.uint64(1)
    return np.where(sh < 64, bit, 0).astype(np.uint8)


def _signed_field(v, bits):
    return np.asarray(v, dtype=np.int64).astype(np.uint64) & np.uint64((1 << bits) - 1)


def _fixed_residual(s, order):
    r = s.astype(np.int64)
    for _ in range(order):
        r = np.diff(r)
    return r


def _lpc_coefs(s, order, precision, shift):
    """Quantised least-squares predictor (any coefficients decode; good ones keep the residual small)."""
    x = s.astype(np.float64)
    n = len(x)
    if n > order + 1:
        a = np.stack([x[order - 1 - j:n - 1 - j] for j in range(order)], axis=1)
        c, *_ = np.linalg.lstsq(a, x[order:], rcond=None)
    else:
        c = np.zeros(order)
    lim = (1 << (precision - 1)) - 1
    if shift is None:
        m = np.max(np.abs(c)) if c.size else 0.0
        shift = 0
        while shift < 15 and m * (1 << (shift + 1)) <= lim:
            shift += 1
    q = np.clip(np.round(c * (1 << shift)), -lim - 1, lim).astype(np.int64)
    return q, shift


def _lpc_residual(s, q, shift):
    s = s.astype(np.int64)
    order = len(q)
    acc = np.zeros(len(s) - order, dtype=np.int64)
    for j in range(order):
        acc += q[j] * s[order - 1 - j:len(s) - 1 - j]
    return s[order:] - (acc >> shift)


def _residual_fields(r, block, order, sub):
    vals, nb = [sub.method, 0], [2, 4]
    po = sub.porder
    if po is None:
        po = 0
        while po < 4 and block % (1 << (po + 1)) == 0 and (block >> (po + 1)) >= order:
            po += 1
    vals[1] = po
    parts = 1 << po
    psz = block >> po
    pbits = 5 if sub.method else 4
    esc = (1 << pbits) - 1
    kmax = esc - 1
    out_v, out_n = [np.array(vals, np.uint64)], [np.array(nb, np.int64)]
    i = 0
    for p in range(parts):
        n = psz - order if p == 0 else psz
        part = r[i:i + n]
        i += n
        if p in sub.escape:
            w = sub.escape_width
            if w is None:
                m = int(np.max(np.abs(part))) if n else 0
                w = int(m).bit_length() + 1 if m else 0
            out_v.append(np.array([esc, w], np.uint64))
            out_n.append(np.array([pbits, 5], np.int64))
            if w:
                out_v.append(_signed_field(part, w))
                out_n.append(np.full(n, w, np.int64))
            continue
        u = np.where(part >= 0, 2 * part, -2 * part - 1).astype(np.int64)
        if sub.rice is not None:
            k = sub.rice
        else:
            mean = float(u.mean()) if n else 0.0
            k = int(np.clip(np.floor(np.log2(mean + 1)), 0, kmax)) if mean > 0 else 0
        out_v.append(np.array([k], np.uint64))
        out_n.append(np.array([pbits], np.int64))
        if n:
            q = u >> k
            low = u & ((1 << k) - 1)
            out_v.append(((np.uint64(1) << np.uint64(k)) | low.astype(np.uint64)))
            out_n.append(q + 1 + k)
    return np.concatenate(out_v), np.concatenate(out_n)


def encode_subframe(s, bps, sub):
    """Fields (values, widths) of one subframe of the int samples s at bps bits."""
    s = np.asarray(s, dtype=np.int64)
    block = len(s)
    k = sub.wasted
    if k:
        assert not np.any(s & ((1 << k) - 1)), "samples are not multiples of 2^wasted"
        s = s >> k
        bps -= k
    head_v, head_n = [], []
    if sub.kind == "constant":
        assert np.all(s == s[0])
        t = 0
    elif sub.kind == "verbatim":
        t = 1
    elif sub.kind == "fixed":
        assert 0 <= sub.order <= 4 and sub.order <= block, "FIXED order is 0..4"
        t = 8 + sub.order
    else:
        assert 1 <= sub.order <= 32 and sub.order <= block, "LPC order is 1..32"
        t = 31 + sub.order
    head_v += [0, t, 1 if k else 0]
    head_n += [1, 6, 1]
    if k:
        head_v.append(1)
        head_n.append(k)                       # k - 1 zeros, then a one
    v, n = [np.array(head_v, np.uint64)], [np.array(head_n, np.int64)]
    if sub.kind == "constant":
        v.append(_signed_field([s[0]], bps))
        n.append(np.array([bps]))
    elif sub.kind == "verbatim":
        v.append(_signed_field(s, bps))
        n.append(np.full(block, bps))
    elif sub.kind == "fixed":
        o = sub.order
        v.append(_signed_field(s[:o], bps))
        n.append(np.full(o, bps))
        rv, rn = _residual_fields(_fixed_residual(s, o), block, o, sub)
        v.append(rv)
        n.append(rn)
    else:
        o = sub.order
        precision = sub.precision or 12
        q, shift = _lpc_coefs(s, o, precision, sub.shift)
        v.append(_signed_field(s[:o], bps))
        n.append(np.full(o, bps))
        v.append(np.array([precision - 1], np.uint64))
        n.append(np.array([4]))
        v.append(_signed_field([shift], 5))
        n.append(np.array([5]))
        v.append(_signed_field(q, precision))
        n.append(np.full(o, precision))
        rv, rn = _residual_fields(_lpc_residual(s, q, shift), block, o, sub)
        v.append(rv)
        n.append(rn)
    return np.concatenate(v), np.concatenate(n).astype(np.int64)


def frame_header(block, number, variable, rate, bits, channels, assignment, bs_code=None, rate_code=None,
                 size_code=None):
    if bs_code is None:
        common = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5}
        common.update({256 << i: 8 + i for i in range(8)})
        bs_code = common.get(block, 6 if block <= 256 else 7)
    if rate_code is None:
        rate_code = RATE_CODES.get(rate)
        if rate_code is None:
            rate_code = 12 if rate % 1000 == 0 and rate // 1000 < 256 else 13 if rate < 65536 else 14
    if size_code is None:
        size_code = SIZE_CODES[bits]
    ch_code = assignment if assignment >= 8 else channels - 1
    h = bytearray([0xFF, 0xF8 | variable, (bs_code << 4) | rate_code, (ch_code << 4) | (size_code << 1)])
    h += utf8_number(number)
    if bs_code == 6:
        h.append(block - 1)
    elif bs_code == 7:
        h += (block - 1).to_bytes(2, "big")
    if rate_code == 12:
        h.append(rate // 1000)
    elif rate_code == 13:
        h += rate.to_bytes(2, "big")
    elif rate_code == 14:
        h += (rate // 10).to_bytes(2, "big")
    h.append(crc8(h))
    return bytes(h)


def encode_frame(x, bits, rate, number, variable=False, stereo="independent", sub=None, header=None):
    """One frame of x [block, channels] (int).  sub: a Sub, or a list of one per channel."""
    block, channels = x.shape
    assignment = STEREO[stereo] if channels == 2 else 1
    x = x.astype(np.int64)
    if channels == 2 and assignment != 1:
        l, r = x[:, 0], x[:, 1]
        if assignment == 8:
            chans, widths = [l, l - r], [bits, bits + 1]
        elif assignment == 9:
            chans, widths = [l - r, r], [bits + 1, bits]
        else:
            chans, widths = [(l + r) >> 1, l - r], [bits, bits + 1]
    else:
        chans, widths = [x[:, c] for c in range(channels)], [bits] * channels
    subs = sub if isinstance(sub, (list, tuple)) else [sub or Sub()] * channels
    hdr = frame_header(block, number, int(variable), rate, bits, channels, assignment, **(header or {}))
    v, n = zip(*(encode_subframe(c, w, s) for c, w, s in zip(chans, widths, subs)))
    body = _fields_to_bits(np.concatenate(v), np.concatenate(n))
    body = np.concatenate([body, np.zeros((-body.size) % 8, np.uint8)])
    frame = hdr + np.packbits(body).tobytes()
    return frame + crc16(frame).to_bytes(2, "big")


def streaminfo(rate, channels, bits, total, min_block, max_block):
    v = (min_block << 128) | (max_block << 112) | (rate << 44) | ((channels - 1) << 41) | ((bits - 1) << 36) | total
    return v.to_bytes(18, "big") + bytes(16)


def metadata_block(kind, body, last):
    return bytes([(0x80 if last else 0) | kind]) + len(body).to_bytes(3, "big") + body


def encode(x, rate, bits, block=4096, blocks=None, variable=False, stereo="independent", sub=None, metadata=(),
           header=None, info=None):
    """FLAC stream of x [n, channels] (ints of `bits` bits).  blocks: explicit block sizes (else `block`, the last
    frame shorter); stereo / sub / header: a value for every frame or a callable f(frame index) -> value; metadata:
    (type, body) blocks after STREAMINFO; info: STREAMINFO field overrides (min_block, max_block, total, rate,
    channels, bits)."""
    x = np.asarray(x)
    if x.ndim == 1:
        x = x[:, None]
    n, channels = x.shape
    if blocks is None:
        blocks = [block] * (n // block) + ([n % block] if n % block else [])
    assert sum(blocks) == n
    pick = (lambda v, i: v(i) if callable(v) else v)
    frames, at = [], 0
    for i, b in enumerate(blocks):
        frames.append(encode_frame(x[at:at + b], bits, rate, at if variable else i, variable, pick(stereo, i),
                                   pick(sub, i), pick(header, i)))
        at += b
    si = dict(min_block=min(blocks), max_block=max(blocks), total=n, rate=rate, channels=channels, bits=bits)
    si.update(info or {})
    blocks_meta = [(0, streaminfo(si["rate"], si["channels"], si["bits"], si["total"], si["min_block"],
                                  si["max_block"]))] + list(metadata)
    out = bytearray(b"fLaC")
    for i, (kind, body) in enumerate(blocks_meta):
        out += metadata_block(kind, body, i == len(blocks_meta) - 1)
    for f in frames:
        out += f
    return bytes(out)


# ---- decoder ---------------------------------------------------------------------------------------------------
class _Bits:
    def __init__(self, data, pos):
        self.b = np.unpackbits(np.frombuffer(data, np.uint8)).tolist()
        self.p = pos * 8

    def u(self, n):
        if self.p + n > len(self.b):
            raise EOFError
        v = 0
        for bit in self.b[self.p:self.p + n]:
            v = (v << 1) | bit
        self.p += n
        return v

    def s(self, n):
        if n == 0:
            return 0
        v = self.u(n)
        return v - (1 << n) if v >> (n - 1) else v

    def unary(self):
        try:
            i = self.b.index(1, self.p)
        except ValueError:
            raise EOFError from None
        q = i - self.p
        self.p = i + 1
        return q


def _residual(br, block, order):
    method = br.u(2)
    assert method < 2, "reserved residual method"
    pbits = 5 if method else 4
    po = br.u(4)
    psz = block >> po
    assert block % (1 << po) == 0 and psz >= order, "bad partition order"
    out = []
    for p in range(1 << po):
        n = psz - order if p == 0 else psz
        k = br.u(pbits)
        if k == (1 << pbits) - 1:
            w = br.u(5)
            out += [br.s(w) for _ in range(n)]
        else:
            for _ in range(n):
                u = (br.unary() << k) | br.u(k)
                out.append((u >> 1) ^ -(u & 1))
    return out


def _subframe(br, bps, block):
    assert br.u(1) == 0, "subframe padding bit"
    t = br.u(6)
    k = br.unary() + 1 if br.u(1) else 0
    bps -= k
    if t == 0:
        s = [br.s(bps)] * block
    elif t == 1:
        s = [br.s(bps) for _ in range(block)]
    elif 8 <= t <= 12:
        o = t - 8
        s = [br.s(bps) for _ in range(o)]
        coefs = [[], [1], [2, -1], [3, -3, 1], [4, -6, 4, -1]][o]
        for r in _residual(br, block, o):
            s.append(r + sum(c * s[-1 - j] for j, c in enumerate(coefs)))
    elif t >= 32:
        o = t - 31
        s = [br.s(bps) for _ in range(o)]
        prec = br.u(4) + 1
        assert prec != 16, "invalid LPC precision"
        shift = br.s(5)
        assert shift >= 0, "negative LPC shift"
        q = [br.s(prec) for _ in range(o)]
        for r in _residual(br, block, o):
            s.append(r + (sum(c * s[-1 - j] for j, c in enumerate(q)) >> shift))
    else:
        raise AssertionError("reserved subframe type")
    return [v << k for v in s]


def decode_frame(data, pos, bits, channels, rate):
    """One frame at data[pos]: dict of header fields, 'end' and 'samples' [block, channels] (int64)."""
    d = data
    assert d[pos] == 0xFF and d[pos + 1] & 0xFE == 0xF8, "no sync"
    variable = d[pos + 1] & 1
    bs_code, sr_code, ch_code, ss_code = d[pos + 2] >> 4, d[pos + 2] & 15, d[pos + 3] >> 4, (d[pos + 3] >> 1) & 7
    q = pos + 4
    c0 = d[q]
    n, v = 0, c0
    if c0 >= 0x80:
        while (c0 << n) & 0x80:                # leading ones: bytes of the number
            n += 1
        v = c0 & (0xFF >> (n + 1))
        n -= 1
    q += 1
    for _ in range(n):
        v = (v << 6) | (d[q] & 0x3F)
        q += 1
    block = {1: 192}.get(bs_code)
    if 2 <= bs_code <= 5:
        block = 576 << (bs_code - 2)
    elif bs_code == 6:
        block = d[q] + 1
        q += 1
    elif bs_code == 7:
        block = int.from_bytes(d[q:q + 2], "big") + 1
        q += 2
    elif bs_code >= 8:
        block = 256 << (bs_code - 8)
    if sr_code == 12:
        frate = d[q] * 1000
        q += 1
    elif sr_code in (13, 14):
        frate = int.from_bytes(d[q:q + 2], "big") * (10 if sr_code == 14 else 1)
        q += 2
    else:
        frate = rate if sr_code == 0 else {c: r for r, c in RATE_CODES.items()}[sr_code]
    assert crc8(d[pos:q]) == d[q], "header CRC-8"
    fbits = bits if ss_code == 0 else {c: b for b, c in SIZE_CODES.items()}[ss_code]
    nch = ch_code + 1 if ch_code < 8 else 2
    br = _Bits(d, q + 1)
    subs = []
    for c in range(nch):
        side = (ch_code == 8 and c == 1) or (ch_code == 9 and c == 0) or (ch_code == 10 and c == 1)
        subs.append(_subframe(br, fbits + side, block))
    br.p = (br.p + 7) // 8 * 8
    end = br.p // 8 + 2
    assert crc16(d[pos:end - 2]) == int.from_bytes(d[end - 2:end], "big"), "frame CRC-16"
    a, b = (np.array(subs[0], np.int64), np.array(subs[1], np.int64)) if nch == 2 else (None, None)
    if ch_code == 8:
        subs = [a, a - b]
    elif ch_code == 9:
        subs = [a + b, b]
    elif ch_code == 10:
        m = (a << 1) | (b & 1)
        subs = [(m + b) >> 1, (m - b) >> 1]
    return dict(number=v, block=block, variable=variable, assignment=ch_code, channels=nch, bits=fbits, rate=frate,
                end=end, samples=np.stack([np.asarray(s, np.int64) for s in subs], axis=1))


def decode(data):
    """(samples [n, channels] int64, rate, bits, frames: list of (start, decode_frame dict))."""
    assert data[:4] == b"fLaC"
    pos, last, info = 4, False, None
    while not last:
        last, kind, n = data[pos] >> 7, data[pos] & 0x7F, int.from_bytes(data[pos + 1:pos + 4], "big")
        if kind == 0:
            info = int.from_bytes(data[pos + 4:pos + 22], "big")
        pos += 4 + n
    rate, channels = (info >> 44) & 0xFFFFF, ((info >> 41) & 7) + 1
    bits, total = ((info >> 36) & 31) + 1, info & ((1 << 36) - 1)
    out, frames, got = [], [], 0
    while got < total:
        f = decode_frame(data, pos, bits, channels, rate)
        frames.append((pos, f))
        out.append(f["samples"])
        got += f["block"]
        pos = f["end"]
    return np.concatenate(out), rate, bits, frames


def wav_bytes(x, rate, bits):
    """RIFF/WAVE file holding the int samples x [n, channels] (u8 v + 128, i16, packed i24)."""
    x = np.asarray(x, np.int64)
    if x.ndim == 1:
        x = x[:, None]
    channels = x.shape[1]
    if bits == 8:
        data = (x + 128).astype(np.uint8).tobytes()
    elif bits == 16:
        data = x.astype("<i2").tobytes()
    else:
        data = x.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    nb = bits // 8
    fmt = (1).to_bytes(2, "little") + channels.to_bytes(2, "little") + rate.to_bytes(4, "little") + \
        (rate * channels * nb).to_bytes(4, "little") + (channels * nb).to_bytes(2, "little") + bits.to_bytes(2, "little")
    body = b"WAVE" + b"fmt " + len(fmt).to_bytes(4, "little") + fmt + b"data" + len(data).to_bytes(4, "little") + data
    if len(data) & 1:
        body += b"\0"
    return b"RIFF" + len(body).to_bytes(4, "little") + body
