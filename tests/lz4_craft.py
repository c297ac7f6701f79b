"""LZ4 streams written sequence by sequence, and a strict reader for them.

The writer takes exact sequences — (literals, offset, match length) plus the final literals — with no compressor in
between, so a test can aim at any length chain, offset or block size the format allows, including streams that break its
rules on purpose. `frame()` returns the stream together with the bytes it decodes to (None when no decoder may accept it).

`check_block()` / `check_stream()` take a block or a stream back to its sequences and report the first rule it breaks,
with liblz4's limits (lz4.c: MINMATCH 4, LASTLITERALS 5, MFLIMIT 12; lz4frame.c: header and block size checks).

`liblz4()` is liblz4 through ctypes (LZ4_decompress_safe); whole streams go through oracle.Standin (LZ4F_decompress)."""
import ctypes
import struct
from dataclasses import dataclass, field

FRAME_MAGIC = 0x184D2204
SKIPPABLE_MAGIC = 0x184D2A50
STORED = 0x80000000
LAST_LITERALS = 5
MF_LIMIT = 12
BLOCK_MAX = {4: 64 << 10, 5: 256 << 10, 6: 1 << 20, 7: 4 << 20}


def xxh32(data: bytes, seed: int = 0) -> int:
    P1, P2, P3, P4, P5, M = 2654435761, 2246822519, 3266489917, 668265263, 374761393, 0xFFFFFFFF
    rot = lambda x, r: ((x << r) | (x >> (32 - r))) & M
    n, i = len(data), 0
    if n >= 16:
        v = [(seed + P1 + P2) & M, (seed + P2) & M, seed & M, (seed - P1) & M]
        words = struct.unpack_from("<%dI" % (4 * (n // 16)), data)
        for k, w in enumerate(words):
            v[k & 3] = (rot((v[k & 3] + w * P2) & M, 13) * P1) & M
        i = 16 * (n // 16)
        h = (rot(v[0], 1) + rot(v[1], 7) + rot(v[2], 12) + rot(v[3], 18)) & M
    else:
        h = (seed + P5) & M
    h = (h + n) & M
    while i + 4 <= n:
        h = (rot((h + struct.unpack_from("<I", data, i)[0] * P3) & M, 17) * P4) & M
        i += 4
    while i < n:
        h = (rot((h + data[i] * P5) & M, 11) * P1) & M
        i += 1
    h ^= h >> 15
    h = (h * P2) & M
    h ^= h >> 13
    h = (h * P3) & M
    return h ^ (h >> 16)


# ------------------------------------------------------------------------------------------------ writer
def _chain(n: int) -> bytes:
    """the length bytes behind a nibble of 15: n more, as 255s and a final byte < 255"""
    return b"\xff" * (n // 255) + bytes([n % 255])


def encode_block(seqs, final=b""):
    """seqs: (literals, offset, match_len) in stream order; final: the literals of the last sequence, None for a block
    that ends with a match (which breaks the end rules)"""
    out = bytearray()
    for lit, off, ml in seqs:
        assert ml >= 4 and 0 <= off <= 0xFFFF
        tl, tm = min(len(lit), 15), min(ml - 4, 15)
        out.append(tl << 4 | tm)
        if tl == 15:
            out += _chain(len(lit) - 15)
        out += lit
        out += struct.pack("<H", off)
        if tm == 15:
            out += _chain(ml - 19)
    if final is not None:
        tl = min(len(final), 15)
        out.append(tl << 4)
        if tl == 15:
            out += _chain(len(final) - 15)
        out += final
    return bytes(out)


def expand(seqs, final, window=b""):
    """the bytes a block decodes to, behind `window` (the frame's output in front of it); None when a match has offset 0
    or reaches in front of the window"""
    out = bytearray(window)
    for lit, off, ml in seqs:
        out += lit
        if off == 0 or off > len(out):
            return None
        src = out[len(out) - off:len(out) - off + ml]
        if off < ml:
            src = (src * (ml // off + 1))[:ml]
        out += src
    out += final or b""
    return bytes(out[len(window):])


@dataclass
class Block:
    """a compressed block (seqs + final) or, with `stored`, a stored one"""
    seqs: list = field(default_factory=list)
    final: bytes = b""
    stored: bytes = None

    def data(self):
        return self.stored if self.stored is not None else encode_block(self.seqs, self.final)


def frame(blocks, linked=False, bsid=4, block_checksum=False, content_checksum=False, content_size=False, dict_id=None,
          version=1, endmark=True):
    """one LZ4 frame -> (stream bytes, decoded bytes or None)"""
    flg = version << 6 | (0 if linked else 1) << 5 | block_checksum << 4 | content_size << 3 | content_checksum << 2
    flg |= dict_id is not None
    out, body = bytearray(), bytearray()
    ok = True
    for b in blocks:
        data = b.data()
        out += struct.pack("<I", len(data) | (STORED if b.stored is not None else 0)) + data
        if block_checksum:
            out += struct.pack("<I", xxh32(data))
        if not ok:
            continue
        got = b.stored if b.stored is not None else expand(b.seqs, b.final, bytes(body[-65535:]) if linked else b"")
        if got is None:
            ok = False
        else:
            body += got
    desc = bytes([flg & 0xFF, (bsid & 7) << 4])
    if content_size:
        desc += struct.pack("<Q", len(body))
    if dict_id is not None:
        desc += struct.pack("<I", dict_id)
    head = struct.pack("<I", FRAME_MAGIC) + desc + bytes([(xxh32(desc) >> 8) & 0xFF])
    tail = struct.pack("<I", 0) if endmark else b""
    if endmark and content_checksum:
        tail += struct.pack("<I", xxh32(bytes(body)))
    return head + bytes(out) + tail, (bytes(body) if ok else None)


def skippable(payload=b"", nibble=0):
    return struct.pack("<II", SKIPPABLE_MAGIC | nibble, len(payload)) + payload, b""


def stream(*parts):
    """concatenates (bytes, decoded) pairs; decoded is None when any part is"""
    data = b"".join(p[0] for p in parts)
    dec = None if any(p[1] is None for p in parts) else b"".join(p[1] for p in parts)
    return data, dec


# ------------------------------------------------------------------------------------------------ strict reader
class Broken(Exception):
    pass


def parse_block(data):
    """a compressed block -> (seqs, final); final is None when the block ends with a match. Raises Broken when a length
    chain, a literal run or an offset runs off the block."""
    seqs, ip, n = [], 0, len(data)
    while ip < n:
        token = data[ip]
        ip += 1
        lit = token >> 4
        if lit == 15:
            while True:
                if ip >= n:
                    raise Broken("literal length chain runs off the block")
                lit += data[ip]
                ip += 1
                if data[ip - 1] != 255:
                    break
        if ip + lit > n:
            raise Broken("literal run past the block end")
        lits = bytes(data[ip:ip + lit])
        ip += lit
        if ip == n:
            return seqs, lits
        if ip + 2 > n:
            raise Broken("offset past the block end")
        off = data[ip] | data[ip + 1] << 8
        ip += 2
        ml = token & 15
        if ml == 15:
            while True:
                if ip >= n:
                    raise Broken("match length chain runs off the block")
                ml += data[ip]
                ip += 1
                if data[ip - 1] != 255:
                    break
        seqs.append((lits, off, ml + 4))
    return seqs, None


def check_block(data, window=0, raw_max=None):
    """the first LZ4 rule a compressed block breaks, or None. window: bytes of the frame in front of the block (0 for an
    independent block); raw_max: the frame's block maximum"""
    try:
        seqs, final = parse_block(data)
    except Broken as e:
        return str(e)
    op = last_match = 0
    for k, (lit, off, ml) in enumerate(seqs):
        op += len(lit)
        if off == 0:
            return f"sequence {k}: offset 0"
        if off > op + window:
            return f"sequence {k}: offset {off} reaches in front of the {'frame' if window else 'block'}"
        last_match = op
        op += ml
    if final is None:
        return "the block ends with a match"
    op += len(final)
    if seqs and len(final) < LAST_LITERALS:
        return f"a match touches the last {LAST_LITERALS} bytes ({len(final)} final literals)"
    if seqs and op - last_match < MF_LIMIT:
        return f"the last match starts {op - last_match} bytes before the block end"
    if raw_max is not None and op > raw_max:
        return f"decoded size {op} above the block maximum {raw_max}"
    return None


@dataclass
class FrameInfo:
    flg: int
    bd: int
    linked: bool
    block_max: int
    content_size: int
    dict_id: int
    words: list          # block header words, in order
    raw: list            # decoded size of every block


def check_stream(data, shrink=True):
    """walks a stream of LZ4 and skippable frames -> (decoded bytes, [FrameInfo]); raises Broken at the first broken
    rule. With `shrink`, a compressed block must be smaller than its raw size (an encoder stores it otherwise)."""
    pos, out, frames = 0, bytearray(), []
    rd = lambda p, n: int.from_bytes(data[p:p + n], "little")
    while pos < len(data):
        if pos + 8 > len(data):
            raise Broken("truncated frame header")
        magic = rd(pos, 4)
        if magic & 0xFFFFFFF0 == SKIPPABLE_MAGIC:
            pos += 8 + rd(pos + 4, 4)
            if pos > len(data):
                raise Broken("truncated skippable frame")
            continue
        if magic != FRAME_MAGIC:
            raise Broken(f"bad magic at {pos}")
        flg, bd = data[pos + 4], data[pos + 5]
        if flg >> 6 != 1 or flg & 2 or bd & 0x8F or (bd >> 4) & 7 < 4:
            raise Broken("bad frame descriptor")
        hlen = 2 + (8 if flg & 8 else 0) + (4 if flg & 1 else 0)
        desc = bytes(data[pos + 4:pos + 4 + hlen])
        if data[pos + 4 + hlen] != (xxh32(desc) >> 8) & 0xFF:
            raise Broken("bad header checksum")
        info = FrameInfo(flg, bd, not (flg & 0x20), BLOCK_MAX[(bd >> 4) & 7], rd(pos + 6, 8) if flg & 8 else None,
                         rd(pos + 6 + (8 if flg & 8 else 0), 4) if flg & 1 else None, [], [])
        p, body = pos + 5 + hlen, bytearray()
        while True:
            if p + 4 > len(data):
                raise Broken("truncated block header")
            word = rd(p, 4)
            p += 4
            if word == 0:
                break
            size = word & ~STORED
            if size > info.block_max or p + size > len(data):
                raise Broken(f"block of {size} bytes at {p}")
            blk = bytes(data[p:p + size])
            if word & STORED:
                got = blk
            else:
                window = bytes(body[-65535:]) if info.linked else b""
                problem = check_block(blk, len(window), info.block_max)
                if problem:
                    raise Broken(f"block {len(info.words)} of frame {len(frames)}: {problem}")
                got = expand(*parse_block(blk), window)
                if shrink and size >= len(got):
                    raise Broken(f"compressed block {len(info.words)} of frame {len(frames)} is not smaller than raw")
            info.words.append(word)
            info.raw.append(len(got))
            body += got
            p += size + (4 if flg & 0x10 else 0)
        if flg & 4:
            if rd(p, 4) != xxh32(bytes(body)):
                raise Broken("content checksum")
            p += 4
        if info.content_size is not None and info.content_size != len(body):
            raise Broken("content size")
        out += body
        frames.append(info)
        pos = p
    return bytes(out), frames


# ------------------------------------------------------------------------------------------------ liblz4
_lib = None


def liblz4():
    """liblz4 with LZ4_decompress_safe declared; None where the library is missing"""
    global _lib
    if _lib is None:
        try:
            L = ctypes.CDLL("liblz4.so.1")
        except OSError:
            return None
        L.LZ4_decompress_safe.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
        L.LZ4_decompress_safe.restype = ctypes.c_int
        _lib = L
    return _lib


def decompress_block(data, capacity):
    """LZ4_decompress_safe on one block with room for exactly `capacity` bytes: decoded size, or < 0 when refused"""
    dst = ctypes.create_string_buffer(max(capacity, 1))
    return liblz4().LZ4_decompress_safe(bytes(data), dst, len(data), capacity)
