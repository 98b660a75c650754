"""FLAC test helpers: a deliberate FLAC writer and an independent decoder (FFmpeg's libavcodec, through ctypes).

The writer emits exactly the stream it is asked for -- every subframe type (CONSTANT, VERBATIM, FIXED 0-4, LPC 1-32
with any precision and shift), wasted bits, Rice and Rice2 residuals with any partition order, escaped partitions,
all channel assignments, every block-size and sample-rate code, fixed and variable blocking, ID3v2 tags and extra
metadata blocks -- so that tests can reach every path of the decoder.  Its output is checked against FFmpeg, which
shares no code with the package, before it is used as a reference.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import struct
import sys

import numpy as np

# ---- bits ----------------------------------------------------------------------------------------------------------


class BitWriter:
    """MSB-first bit fields, packed with numpy (a field wider than 64 bits holds a value below 2^64: unary codes)."""

    def __init__(self):
        self.vals, self.widths = [], []
        self.nbits = 0

    def put(self, v: int, n: int):
        self.put_many(np.array([int(v) & ((1 << 64) - 1)], np.uint64), np.array([n], np.int64))

    def put_signed(self, v: int, n: int):
        assert -(1 << (n - 1)) <= v < (1 << (n - 1)) if n else v == 0, (v, n)
        self.put(int(v) & ((1 << n) - 1) if n else 0, n)

    def put_many(self, vals, widths):
        vals = np.asarray(vals, np.uint64)
        widths = np.broadcast_to(np.asarray(widths, np.int64), vals.shape)
        self.vals.append(vals)
        self.widths.append(widths)
        self.nbits += int(widths.sum())

    def pad(self):
        if self.nbits % 8:
            self.put(0, 8 - self.nbits % 8)

    def tobytes(self) -> bytes:
        self.pad()
        if not self.vals:
            return b""
        v, w = np.concatenate(self.vals), np.concatenate(self.widths)
        ends = np.cumsum(w)
        bits = np.zeros(int(ends[-1]) if len(ends) else 0, np.uint8)
        for b in range(64):
            m = w > b
            if not m.any():
                break
            bits[ends[m] - 1 - b] = ((v[m] >> np.uint64(b)) & np.uint64(1)).astype(np.uint8)
        return np.packbits(bits).tobytes()


def _crc_table(poly, width):
    top, mask = 1 << (width - 1), (1 << width) - 1
    t = []
    for i in range(256):
        c = i << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
        t.append(c)
    return t


_CRC8, _CRC16 = _crc_table(0x07, 8), _crc_table(0x8005, 16)


def crc8(data: bytes) -> int:
    c = 0
    for b in data:
        c = _CRC8[c ^ b]
    return c


def crc16(data: bytes) -> int:
    c = 0
    t = _CRC16
    for b in data:
        c = ((c << 8) & 0xFFFF) ^ t[(c >> 8) ^ b]
    return c


def utf8_number(v: int) -> bytes:
    """FLAC's UTF-8-like coding of a frame or sample number (up to 36 bits, 1 to 7 bytes)."""
    if v < 0x80:
        return bytes([v])
    for n, lead in ((2, 0xC0), (3, 0xE0), (4, 0xF0), (5, 0xF8), (6, 0xFC), (7, 0xFE)):
        if v < (1 << (5 * n + 1 if n < 7 else 36)):
            out = [0x80 | ((v >> (6 * i)) & 0x3F) for i in range(n - 1)][::-1]
            return bytes([lead | (v >> (6 * (n - 1)))] + out)
    raise ValueError(v)


# ---- encoder -------------------------------------------------------------------------------------------------------

BLOCK_CODES = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13,
               16384: 14, 32768: 15}
RATE_CODES = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10,
              96000: 11}
SIZE_CODES = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6, 32: 7}
FIXED = {0: [], 1: [1], 2: [2, -1], 3: [3, -3, 1], 4: [4, -6, 4, -1]}
ASSIGN = {"left_side": 8, "right_side": 9, "mid_side": 10}


def predict(x: np.ndarray, coefs, shift: int) -> np.ndarray:
    """residual[i] = x[i] - (sum_j coefs[j] * x[i-1-j]) >> shift for i >= order, exact in int64."""
    order = len(coefs)
    acc = np.zeros(len(x) - order, np.int64)
    for j, c in enumerate(coefs):
        acc += np.int64(c) * x[order - 1 - j:len(x) - 1 - j]
    return x[order:] - (acc >> shift)


def lpc_coefs(x: np.ndarray, order: int, precision: int, shift=None):
    """Quantised LPC coefficients (Levinson-Durbin on the windowed autocorrelation) and their shift."""
    y = x.astype(np.float64) * np.hanning(len(x) + 2)[1:-1]
    r = np.array([np.dot(y[:len(y) - k], y[k:]) for k in range(order + 1)])
    r[0] = r[0] * (1 + 1e-9) + 1e-9
    a = np.zeros(order)
    err = r[0]
    for i in range(order):
        k = (r[i + 1] - np.dot(a[:i], r[i:0:-1])) / err
        a[:i] = a[:i] - k * a[:i][::-1]
        a[i] = k
        err *= 1 - k * k
        if err <= 0:
            break
    top = np.max(np.abs(a))
    if shift is None:
        shift = 15 if top == 0 else int(np.clip(precision - 2 - np.floor(np.log2(top)), 0, 15))
    lim = 1 << (precision - 1)
    q = np.clip(np.round(a * (1 << shift)), -lim, lim - 1).astype(np.int64)
    return [int(c) for c in q], shift


def _zigzag(r: np.ndarray) -> np.ndarray:
    r = r.astype(np.int64)
    return ((r << 1) ^ (r >> 63)).astype(np.uint64)


def _rice_k(u: np.ndarray, kmax: int) -> int:
    if not len(u):
        return 0
    costs = [int(np.sum(u >> np.uint64(k))) + len(u) * (k + 1) for k in range(kmax + 1)]
    return int(np.argmin(costs))


def _residual(w: BitWriter, res: np.ndarray, n: int, order: int, spec: dict):
    method = spec.get("method")
    if method is None:                                    # Rice2 when a parameter above 14 is cheaper
        method = int(_rice_k(_zigzag(res), 30) > 14)
    kmax, escape = (14, 15) if method == 0 else (30, 31)
    porder = spec.get("porder")
    if porder is None:                                    # the cheapest order the block allows, up to 8
        best = None
        for po in range(0, 9):
            if n % (1 << po) or (n >> po) < order:
                break
            cost = 0
            for p in range(1 << po):
                lo, hi = max(p * (n >> po) - order, 0), (p + 1) * (n >> po) - order
                u = _zigzag(res[lo:hi])
                k = _rice_k(u, kmax)
                cost += int(np.sum(u >> np.uint64(k))) + len(u) * (k + 1)
            if best is None or cost < best[0]:
                best = (cost, po)
        porder = best[1]
    while not spec.get("exact_porder") and porder and (n % (1 << porder) or (n >> porder) < order):
        porder -= 1                                       # what a short last frame allows (exact_porder: as asked)
    w.put(spec.get("method_code", method), 2)             # method_code: a reserved code on request
    w.put(porder, 4)
    psize = n >> porder
    escaped = spec.get("escape", ())
    for p in range(1 << porder):
        lo, hi = max(p * psize - order, 0), (p + 1) * psize - order
        part = res[lo:hi]
        if escaped == "all" or p in escaped:
            nb = spec.get("escape_bits")
            if nb is None:
                m = int(np.max(np.abs(part))) if len(part) else 0
                nb = 0 if m == 0 and (not len(part) or np.all(part == 0)) else int(max(m, 1)).bit_length() + 1
            w.put(escape, 4 if method == 0 else 5)
            w.put(nb, 5)
            if nb:
                w.put_many(part.astype(np.int64).astype(np.uint64) & np.uint64((1 << nb) - 1), nb)
            continue
        u = _zigzag(part)
        k = spec.get("k", _rice_k(u, kmax))
        w.put(k, 4 if method == 0 else 5)
        q = u >> np.uint64(k)
        vals = np.empty(2 * len(u), np.uint64)
        wid = np.empty(2 * len(u), np.int64)
        vals[0::2], wid[0::2] = 1, q.astype(np.int64) + 1
        vals[1::2], wid[1::2] = u & np.uint64((1 << k) - 1), k
        w.put_many(vals, wid)


def subframe(w: BitWriter, x: np.ndarray, sbps: int, spec: dict):
    """One subframe of the integers x (sbps bits each) as spec says: kind constant / verbatim / fixed / lpc, order,
    precision, shift, coefs, wasted, and the residual's method, porder, k, escape, escape_bits."""
    kind = spec.get("kind", "lpc")
    if kind in ("fixed", "lpc") and spec.get("order", 8) > len(x):   # a short last frame cannot hold the warm-up samples
        kind = "verbatim"
    wasted = spec.get("wasted", 0)
    if wasted:
        assert np.all(x % (1 << wasted) == 0)
        x = x >> wasted
    bps = sbps - wasted
    n = len(x)
    w.put(0, 1)
    if "type_code" in spec:                               # a reserved type on request, then verbatim data
        w.put(spec["type_code"], 6)
        kind = "verbatim"
    elif kind == "constant":
        assert np.all(x == x[0])
        w.put(0, 6)
    elif kind == "verbatim":
        w.put(1, 6)
    elif kind == "fixed":
        w.put(8 + spec.get("order", 8), 6)
    else:
        w.put(31 + spec.get("order", 8), 6)
    if wasted:
        w.put(1, 1)
        w.put(1, wasted)                                   # unary wasted - 1: wasted - 1 zeros, then a one
    else:
        w.put(0, 1)
    if kind == "constant":
        w.put_signed(int(x[0]), bps)
        return
    if kind == "verbatim":
        w.put_many(x.astype(np.int64).astype(np.uint64) & np.uint64((1 << bps) - 1), bps)
        return
    order = spec.get("order", 8)
    for v in x[:order]:
        w.put_signed(int(v), bps)
    if kind == "fixed":
        coefs, shift = FIXED[order], 0
    else:
        precision = spec.get("precision", 15)
        if "coefs" in spec:
            coefs, shift = list(spec["coefs"]), spec.get("shift", 0)
        else:
            coefs, shift = lpc_coefs(x, order, precision, spec.get("shift"))
        w.put(precision - 1, 4)
        w.put_signed(shift, 5)
        for c in coefs:
            w.put_signed(c, precision)
    res = predict(x.astype(np.int64), coefs, max(shift, 0))   # a negative shift (invalid) on request: any residual
    assert np.all(np.abs(res) < (1 << 31)), "residual outside 32 bits"
    _residual(w, res, n, order, spec)


def _channels(block: np.ndarray, assignment: str):
    """(coded channels, their bits over the stream's) for an assignment of a [n, C] block."""
    if assignment == "independent":
        return [block[:, c] for c in range(block.shape[1])], [0] * block.shape[1]
    left, right = block[:, 0], block[:, 1]
    side = left - right
    if assignment == "left_side":
        return [left, side], [0, 1]
    if assignment == "right_side":
        return [side, right], [1, 0]
    return [(left + right) >> 1, side], [0, 1]


def frame(x: np.ndarray, bps: int, rate: int, number: int, variable: bool, opts: dict) -> bytes:
    """One frame of the [n, C] integers x.  opts: assignment, subframes (a spec or one per channel), block_code
    ("auto", 6 or 7), rate_code ("auto", 0, 12, 13, 14), size_code ("auto" or 0)."""
    n, nch = x.shape
    h = BitWriter()
    h.put(0xFFF8 | int(variable), 16)
    bc = opts.get("block_code", "auto")
    if bc == "auto":
        bc = BLOCK_CODES.get(n, 6 if n <= 256 else 7)
    h.put(bc, 4)
    rc = opts.get("rate_code", "auto")
    if rc == "auto":
        rc = RATE_CODES.get(rate, 0)
    elif rc == "table":
        rc = RATE_CODES[rate]
    h.put(rc, 4)
    assignment = opts.get("assignment", "independent")
    h.put(ASSIGN.get(assignment, nch - 1), 4)
    sc = opts.get("size_code", "auto")
    h.put(SIZE_CODES.get(bps, 0) if sc == "auto" else sc, 3)
    h.put(0, 1)
    head = h.tobytes() + utf8_number(number)
    if bc == 6:
        head += bytes([n - 1])
    elif bc == 7:
        head += struct.pack(">H", n - 1)
    if rc == 12:
        head += bytes([rate // 1000])
    elif rc == 13:
        head += struct.pack(">H", rate)
    elif rc == 14:
        head += struct.pack(">H", rate // 10)
    head += bytes([crc8(head)])
    w = BitWriter()
    chans, extra = _channels(x, assignment)
    specs = opts.get("subframes", {})
    for c, (xc, e) in enumerate(zip(chans, extra)):
        spec = specs[c] if isinstance(specs, (list, tuple)) else specs
        subframe(w, xc.astype(np.int64), bps + e, spec)
    body = head + w.tobytes()
    return body + struct.pack(">H", crc16(body))


def streaminfo(rate, channels, bps, total, min_block=16, max_block=4096) -> bytes:
    w = BitWriter()
    for v, n in ((min_block, 16), (max_block, 16), (0, 24), (0, 24), (rate, 20), (channels - 1, 3), (bps - 1, 5),
                 (total, 36)):
        w.put(v, n)
    return w.tobytes() + bytes(16)


def id3v2(size: int, footer=False) -> bytes:
    ss = bytes([(size >> 21) & 0x7F, (size >> 14) & 0x7F, (size >> 7) & 0x7F, size & 0x7F])
    body = b"\x00" * size
    return b"ID3\x04\x00" + bytes([0x10 if footer else 0]) + ss + body + (b"3DI\x04\x00\x10" + ss if footer else b"")


class FlacBytes(bytes):
    """A file from encode(); .frames holds each frame's (byte offset, length)."""
    frames: list


def encode(x, rate: int, bps: int, blocks=4096, *, variable=False, first_number=0, opts=None, total="auto",
           metadata=(), id3=None) -> bytes:
    """A FLAC file of the integers x ([n] or [n, C]).  blocks: one block size or a list of them (the last frame takes
    what is left); opts: a dict, or a callable frame index -> dict (see frame()); total: STREAMINFO's sample count
    ("auto": the real one); metadata: extra (type, bytes) blocks after STREAMINFO; id3: an ID3v2 payload size."""
    x = np.asarray(x, np.int64)
    if x.ndim == 1:
        x = x[:, None]
    n, nch = x.shape
    assert -(1 << (bps - 1)) <= x.min() and x.max() < (1 << (bps - 1))
    sizes = []
    at = 0
    while at < n:
        b = blocks if np.isscalar(blocks) else blocks[min(len(sizes), len(blocks) - 1)]
        sizes.append(min(int(b), n - at))
        at += sizes[-1]
    frames = []
    at = 0
    for i, b in enumerate(sizes):
        o = opts(i) if callable(opts) else (opts or {})
        number = first_number + (at if variable else i)
        frames.append(frame(x[at:at + b], bps, rate, number, variable, o))
        at += b
    info = streaminfo(rate, nch, bps, n if total == "auto" else total, max_block=max(sizes + [16]))
    blocks_md = [(0, info)] + list(metadata)
    md = b""
    for j, (t, body) in enumerate(blocks_md):
        md += bytes([(0x80 if j == len(blocks_md) - 1 else 0) | t]) + struct.pack(">I", len(body))[1:] + body
    head = (id3v2(id3) if id3 is not None else b"") + b"fLaC" + md
    out = FlacBytes(head + b"".join(frames))
    out.frames = []
    at = len(head)
    for f in frames:
        out.frames.append((at, len(f)))
        at += len(f)
    return out


# ---- FFmpeg's decoder ----------------------------------------------------------------------------------------------

_FF = None


def _ffmpeg_dir():
    for p in sys.path:
        d = os.path.join(p, "opencv_python_headless.libs")
        if glob.glob(os.path.join(d, "libavcodec-*.so*")):
            return d
    return None


def ffmpeg():
    """libavcodec (with libavutil) from the opencv-python-headless wheel, or None when it is not installed."""
    global _FF
    if _FF is None:
        d = _ffmpeg_dir()
        if d is None:
            _FF = False
            return None
        libs = {}
        try:                                              # dependencies first: libavcodec does not load without libdrm
            for name in ("drm", "crypto", "avutil", "swresample", "vpx", "avcodec"):
                hit = glob.glob(os.path.join(d, f"lib{name}-*.so*"))
                if hit:
                    libs[name] = C.CDLL(hit[0], mode=C.RTLD_GLOBAL)
            av, util = libs["avcodec"], libs["avutil"]
        except (OSError, KeyError):
            _FF = False
            return None
        vp = C.c_void_p
        av.avcodec_find_decoder_by_name.restype = vp
        av.avcodec_alloc_context3.restype = vp
        av.avcodec_alloc_context3.argtypes = [vp]
        av.avcodec_open2.argtypes = [vp, vp, vp]
        av.av_packet_alloc.restype = vp
        av.avcodec_send_packet.argtypes = [vp, vp]
        av.avcodec_receive_frame.argtypes = [vp, vp]
        av.avcodec_free_context.argtypes = [C.POINTER(vp)]
        av.av_packet_free.argtypes = [C.POINTER(vp)]
        util.av_frame_alloc.restype = vp
        util.av_frame_free.argtypes = [C.POINTER(vp)]
        _FF = (av, util)
    return _FF or None


# AVSampleFormat: S16 1, S32 2, S16P 6, S32P 7 -> (bytes per sample, planar)
_FORMATS = {1: (2, False), 2: (4, False), 6: (2, True), 7: (4, True)}


def ffmpeg_decode(data: "FlacBytes", bps: int, channels: int) -> np.ndarray:
    """The [n, channels] int64 samples FFmpeg's FLAC decoder gives for a file written by encode() (metadata as the
    first packet, then one packet per frame, as encode() recorded them).  FFmpeg left-justifies samples in 16- or 32-bit containers; they are
    shifted back by the container width minus bps."""
    av, util = ffmpeg()
    vp = C.c_void_p
    pos = 0
    if data[:3] == b"ID3":
        s = data[6:10]
        pos = 10 + (s[0] << 21 | s[1] << 14 | s[2] << 7 | s[3]) + (10 if data[5] & 0x10 else 0)
    start = pos + 4
    while True:
        last = data[start] & 0x80
        start += 4 + int.from_bytes(data[start + 1:start + 4], "big")
        if last:
            break
    packets = [data[pos:start]] + [data[o:o + n] for o, n in data.frames]
    codec = av.avcodec_find_decoder_by_name(b"flac")
    ctx = vp(av.avcodec_alloc_context3(codec))
    assert av.avcodec_open2(ctx, codec, None) == 0
    pkt, frm = vp(av.av_packet_alloc()), vp(util.av_frame_alloc())
    out = []
    try:
        for chunk in packets:
            buf = C.create_string_buffer(chunk, len(chunk))
            C.c_void_p.from_address(pkt.value + 24).value = C.addressof(buf)
            C.c_int.from_address(pkt.value + 32).value = len(chunk)
            rc = av.avcodec_send_packet(ctx, pkt)
            assert rc == 0, f"avcodec_send_packet: {rc}"
            while av.avcodec_receive_frame(ctx, frm) == 0:
                ns = C.c_int.from_address(frm.value + 112).value
                fmt = C.c_int.from_address(frm.value + 116).value
                size, planar = _FORMATS[fmt]
                ct = C.c_int16 if size == 2 else C.c_int32
                if planar:
                    planes = [np.ctypeslib.as_array((ct * ns).from_address(C.c_void_p.from_address(frm.value + 8 * c).value))
                              for c in range(channels)]
                    y = np.stack(planes, axis=1).astype(np.int64)
                else:
                    y = np.ctypeslib.as_array((ct * (ns * channels)).from_address(C.c_void_p.from_address(frm.value).value))
                    y = y.astype(np.int64).reshape(ns, channels)
                out.append(y >> (8 * size - bps) if bps < 8 * size else y)
        C.c_void_p.from_address(pkt.value + 24).value = None
        C.c_int.from_address(pkt.value + 32).value = 0
    finally:
        av.av_packet_free(C.byref(pkt))
        util.av_frame_free(C.byref(frm))
        av.avcodec_free_context(C.byref(ctx))
    return np.concatenate(out) if out else np.zeros((0, channels), np.int64)
