"""TEST INFRASTRUCTURE ONLY — CPU restatement of the two compression codecs of Kafka record batches that the device
decodes (csrc/ck_inflate.cuh, csrc/ck_lz4.cuh), on top of the framing restatement in oracle/kafka_batch.py.

  * codec 1, gzip: the records section (everything after the 61-byte header) is one gzip member (RFC 1952) around a
    DEFLATE stream (RFC 1951).  Decoded and encoded with the standard library's zlib.
  * codec 3, LZ4: the records section is one LZ4 *frame* (the published "LZ4 Frame Format Description" v1.6.x, magic
    0x184D2204) of LZ4 blocks ("LZ4 Block Format Description"), checksums XXH32 (the published xxHash specification).
    Message format v2 writes the header checksum correctly.  Restated here: XXH32, a frame decoder and a small greedy
    frame encoder covering every flag combination a producer may write.  Pinned by tests/golden/kafka_codecs.json, frames
    written by the system liblz4 (LZ4F_compressFrame), whose content checksums are XXH32 known answers.
  * snappy (2) and zstd (4) are not restated: decode_batches raises on them.
"""
from __future__ import annotations

import base64
import ctypes
import json
import struct
import zlib

from oracle import kafka_batch as kb

NONE, GZIP, SNAPPY, LZ4, ZSTD = 0, 1, 2, 3, 4

# ---- XXH32 ------------------------------------------------------------------------------------------------------------
_P1, _P2, _P3, _P4, _P5 = 2654435761, 2246822519, 3266489917, 668265263, 374761393
_M = 0xFFFFFFFF


def _rotl(x: int, r: int) -> int:
    return ((x << r) | (x >> (32 - r))) & _M


def xxh32(data: bytes, seed: int = 0) -> int:
    n, p = len(data), 0
    if n >= 16:
        v = [(seed + _P1 + _P2) & _M, (seed + _P2) & _M, seed & _M, (seed - _P1) & _M]
        while p + 16 <= n:
            for k in range(4):
                (w,) = struct.unpack_from("<I", data, p + 4 * k)
                v[k] = (_rotl((v[k] + w * _P2) & _M, 13) * _P1) & _M
            p += 16
        h = (_rotl(v[0], 1) + _rotl(v[1], 7) + _rotl(v[2], 12) + _rotl(v[3], 18)) & _M
    else:
        h = (seed + _P5) & _M
    h = (h + n) & _M
    while p + 4 <= n:
        (w,) = struct.unpack_from("<I", data, p)
        h = (_rotl((h + w * _P3) & _M, 17) * _P4) & _M
        p += 4
    while p < n:
        h = (_rotl((h + data[p] * _P5) & _M, 11) * _P1) & _M
        p += 1
    h ^= h >> 15
    h = (h * _P2) & _M
    h ^= h >> 13
    h = (h * _P3) & _M
    h ^= h >> 16
    return h


# ---- LZ4 frame: decode --------------------------------------------------------------------------------------------------
LZ4_MAGIC = 0x184D2204


def _lz4_block(src: bytes, out: bytearray, lo: int, limit: int) -> None:
    ip, n = 0, len(src)
    if not n:
        raise ValueError("empty LZ4 block")
    while True:
        tok = src[ip]
        ip += 1
        lit = tok >> 4
        if lit == 15:
            while True:
                if ip >= n:
                    raise ValueError("literal length runs past the block")
                b = src[ip]
                ip += 1
                lit += b
                if b != 255:
                    break
        if ip + lit > n or len(out) + lit > limit:
            raise ValueError("literals run past the block / output")
        out += src[ip:ip + lit]
        ip += lit
        if ip == n:
            return
        if ip + 2 > n:
            raise ValueError("truncated offset")
        off = src[ip] | src[ip + 1] << 8
        ip += 2
        if off == 0 or off > len(out) - lo:
            raise ValueError(f"offset {off} out of range")
        ml = tok & 15
        if ml == 15:
            while True:
                if ip >= n:
                    raise ValueError("match length runs past the block")
                b = src[ip]
                ip += 1
                ml += b
                if b != 255:
                    break
        ml += 4
        if len(out) + ml > limit:
            raise ValueError("match runs past the block maximum")
        s = len(out) - off
        for k in range(ml):
            out.append(out[s + k])
        if ip >= n:
            raise ValueError("a block must end with literals")


def lz4_frame_decode(src: bytes) -> bytes:
    """one LZ4 frame, all of src (bytes after it are an error)"""
    if len(src) < 7 or struct.unpack_from("<I", src)[0] != LZ4_MAGIC:
        raise ValueError("not an LZ4 frame")
    flg, bd = src[4], src[5]
    if flg >> 6 != 1 or flg & 2 or bd & 0x8F:
        raise ValueError("bad version / reserved bits")
    if flg & 1:
        raise ValueError("DictID frames are not accepted")
    bid = (bd >> 4) & 7
    if bid < 4:
        raise ValueError("bad block maximum")
    bmax = 1 << (8 + 2 * bid)
    indep, bsum, csize, csum = bool(flg & 0x20), bool(flg & 0x10), bool(flg & 0x08), bool(flg & 0x04)
    pos = 6
    stored = None
    if csize:
        (stored,) = struct.unpack_from("<Q", src, pos)
        pos += 8
    if pos >= len(src) or (xxh32(src[4:pos]) >> 8) & 0xFF != src[pos]:
        raise ValueError("header checksum")
    pos += 1
    out = bytearray()
    while True:
        if pos + 4 > len(src):
            raise ValueError("truncated block size")
        (bs,) = struct.unpack_from("<I", src, pos)
        pos += 4
        if bs == 0:
            break
        raw, bs = bool(bs >> 31), bs & 0x7FFFFFFF
        if bs > bmax or pos + bs + (4 if bsum else 0) > len(src):
            raise ValueError("block size")
        blk = src[pos:pos + bs]
        if bsum and xxh32(blk) != struct.unpack_from("<I", src, pos + bs)[0]:
            raise ValueError("block checksum")
        start = len(out)
        if raw:
            out += blk
        else:
            _lz4_block(blk, out, start if indep else 0, start + bmax)
        pos += bs + (4 if bsum else 0)
    if csum:
        if pos + 4 > len(src) or xxh32(bytes(out)) != struct.unpack_from("<I", src, pos)[0]:
            raise ValueError("content checksum")
        pos += 4
    if pos != len(src):
        raise ValueError("bytes after the frame")
    if stored is not None and stored != len(out):
        raise ValueError("content size")
    return bytes(out)


# ---- LZ4 frame: encode (greedy, hash of 4 bytes) -----------------------------------------------------------------------
def _lz4_compress_block(data: bytes, start: int, end: int, window_lo: int) -> bytes:
    """sequences for data[start:end]; matches may reach back to window_lo (>= end - 65535 is kept by the caller)"""
    out = bytearray()
    table: dict[bytes, int] = {}
    for p in range(max(window_lo, start - 65535), start - 3):       # linked blocks: index the preceding window
        table[data[p:p + 4]] = p
    anchor, ip = start, start
    mflimit = end - 12                                              # no match starts in the last 12 bytes
    while ip < mflimit:
        key = data[ip:ip + 4]
        cand = table.get(key)
        table[key] = ip
        if cand is None or ip - cand > 65535 or cand < window_lo:
            ip += 1
            continue
        ml = 4
        while ip + ml < end - 5 and data[cand + ml] == data[ip + ml]:   # the last 5 bytes stay literals
            ml += 1
        _lz4_seq(out, data[anchor:ip], ip - cand, ml)
        for q in range(ip + 1, min(ip + ml, mflimit)):
            table[data[q:q + 4]] = q
        ip += ml
        anchor = ip
    _lz4_seq(out, data[anchor:end], 0, 0)
    return bytes(out)


def _lz4_len(out: bytearray, n: int) -> None:
    while n >= 255:
        out.append(255)
        n -= 255
    out.append(n)


def _lz4_seq(out: bytearray, lit: bytes, off: int, ml: int) -> None:
    m = ml - 4 if ml else 0
    out.append((min(len(lit), 15) << 4) | min(m, 15))
    if len(lit) >= 15:
        _lz4_len(out, len(lit) - 15)
    out += lit
    if not ml:
        return
    out += struct.pack("<H", off)
    if m >= 15:
        _lz4_len(out, m - 15)


def lz4_frame_encode(data: bytes, block_size_id: int = 4, linked: bool = False, block_checksum: bool = False,
                     content_size: bool = False, content_checksum: bool = True, raw_blocks: str = "auto") -> bytes:
    """raw_blocks: "auto" stores a block uncompressed when that is smaller, "all" stores every block uncompressed,
    "odd" stores every second block uncompressed (exercises bit 31 of the block size next to compressed blocks)"""
    bmax = 1 << (8 + 2 * block_size_id)
    flg = 0x40 | (0 if linked else 0x20) | (0x10 if block_checksum else 0) | (0x08 if content_size else 0) | \
        (0x04 if content_checksum else 0)
    desc = bytes([flg, block_size_id << 4]) + (struct.pack("<Q", len(data)) if content_size else b"")
    out = bytearray(struct.pack("<I", LZ4_MAGIC) + desc + bytes([(xxh32(desc) >> 8) & 0xFF]))
    for bi, start in enumerate(range(0, len(data), bmax)):
        end = min(start + bmax, len(data))
        comp = _lz4_compress_block(data, start, end, 0 if linked else start)
        raw = raw_blocks == "all" or (raw_blocks == "odd" and bi % 2 == 1) or len(comp) >= end - start
        blk = data[start:end] if raw else comp
        out += struct.pack("<I", len(blk) | (0x80000000 if raw else 0)) + blk
        if block_checksum:
            out += struct.pack("<I", xxh32(blk))
    out += struct.pack("<I", 0)
    if content_checksum:
        out += struct.pack("<I", xxh32(data))
    return bytes(out)


# ---- gzip ---------------------------------------------------------------------------------------------------------------
def gzip_encode(data: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, mem_level: int = 8,
                fname: bytes | None = None, fextra: bytes | None = None) -> bytes:
    """one gzip member; the header is written here so that FNAME / FEXTRA can be set, the body by zlib (raw deflate)"""
    flg = (4 if fextra is not None else 0) | (8 if fname is not None else 0)
    head = bytearray(b"\x1f\x8b\x08" + bytes([flg]) + b"\0\0\0\0\0\xff")
    if fextra is not None:
        head += struct.pack("<H", len(fextra)) + fextra
    if fname is not None:
        head += fname + b"\0"
    c = zlib.compressobj(level, zlib.DEFLATED, -15, mem_level, strategy)
    body = c.compress(data) + c.flush()
    return bytes(head) + body + struct.pack("<II", zlib.crc32(data), len(data) & _M)


def gzip_decode(src: bytes) -> bytes:
    """exactly one member (bytes after it are an error, as on the device)"""
    d = zlib.decompressobj(31)
    out = d.decompress(src) + d.flush()
    if not d.eof or d.unused_data:
        raise ValueError("not exactly one gzip member")
    return out


# ---- frames -------------------------------------------------------------------------------------------------------------
def frame_with_section(section: bytes, codec: int, count: int, base_offset: int = 0, base_timestamp: int = 0) -> bytes:
    """a RecordBatch v2 frame whose records section is `section` as given (compressed or not), attributes = codec"""
    covered = struct.pack(">hiqqqhii", codec, count - 1, base_timestamp, base_timestamp, -1, -1, -1, count) + section
    return struct.pack(">qiibI", base_offset, len(covered) + 9, 0, 2, kb.crc32c(covered)) + covered


def records_section(records: list[kb.KRecord], base_timestamp: int = 0) -> bytes:
    return bytes(kb.encode_batch(records, base_timestamp=base_timestamp)[kb.HEADER_LEN:])


def encode_batch(records: list[kb.KRecord], base_offset: int = 0, base_timestamp: int = 0, compression: str | None = None,
                 **options) -> bytes:
    """kb.encode_batch with the records section compressed: compression = None, "gzip" (options of gzip_encode) or "lz4"
    (options of lz4_frame_encode)"""
    if compression is None:
        return kb.encode_batch(records, base_offset=base_offset, base_timestamp=base_timestamp)
    plain = records_section(records, base_timestamp)
    if compression == "gzip":
        sec, codec = gzip_encode(plain, **options), GZIP
    elif compression == "lz4":
        sec, codec = lz4_frame_encode(plain, **options), LZ4
    else:
        raise ValueError(f"compression {compression!r} is not restated here")
    max_ts = max([r.timestamp for r in records if r.timestamp] or [base_timestamp])
    f = bytearray(frame_with_section(sec, codec, len(records), base_offset, base_timestamp))
    struct.pack_into(">q", f, 35, max_ts)                         # maxTimestamp, as kb.encode_batch writes it
    struct.pack_into(">I", f, 17, kb.crc32c(bytes(f[kb.CRC_FROM:])))
    return bytes(f)


def load_fixture(path: str) -> list[tuple[dict, bytes, bytes]]:
    """tests/golden/kafka_codecs.json as (case, frame, plaintext records section)"""
    with open(path) as f:
        fx = json.load(f)
    return [(c, base64.b64decode(c["frame"]), zlib.decompress(base64.b64decode(fx["plains"][c["plain"]]))) for c in fx["cases"]]


def decompress_section(codec: int, section: bytes) -> bytes:
    if codec == NONE:
        return section
    if codec == GZIP:
        return gzip_decode(section)
    if codec == LZ4:
        return lz4_frame_decode(section)
    raise ValueError(f"compression codec {codec} is not decoded")


def decode_batches(buf: bytes, verify_crc: bool = True) -> list[kb.KRecord]:
    """kb.decode_batches for fetches that hold gzip / LZ4 frames: every frame's records section is decompressed and
    the records read by the framing restatement"""
    out: list[kb.KRecord] = []
    pos = 0
    while pos + 12 <= len(buf):
        _base, blen = struct.unpack_from(">qi", buf, pos)
        end = pos + 12 + blen
        if end > len(buf):
            break
        f = buf[pos:end]
        if verify_crc and kb.crc32c(f[kb.CRC_FROM:]) != struct.unpack_from(">I", f, 17)[0]:
            raise ValueError("CRC32C mismatch")
        codec = struct.unpack_from(">h", f, kb.CRC_FROM)[0] & 7
        plain = decompress_section(codec, f[kb.HEADER_LEN:])
        g = bytearray(f[:kb.HEADER_LEN] + plain)
        struct.pack_into(">i", g, 8, len(g) - 12)
        struct.pack_into(">h", g, kb.CRC_FROM, struct.unpack_from(">h", f, kb.CRC_FROM)[0] & ~7)
        out += kb.decode_batches(bytes(g), verify_crc=False)
        pos = end
    return out


# ---- the system liblz4, where it exists (fixture generation and a cross-check; no test needs it) -------------------------
class _Prefs(ctypes.Structure):         # LZ4F_preferences_t: LZ4F_frameInfo_t, then the compression settings
    _fields_ = [("blockSizeID", ctypes.c_int), ("blockMode", ctypes.c_int), ("contentChecksumFlag", ctypes.c_int),
                ("frameType", ctypes.c_int), ("contentSize", ctypes.c_ulonglong), ("dictID", ctypes.c_uint),
                ("blockChecksumFlag", ctypes.c_int), ("compressionLevel", ctypes.c_int), ("autoFlush", ctypes.c_uint),
                ("favorDecSpeed", ctypes.c_uint), ("reserved", ctypes.c_uint * 3)]


def liblz4():
    """the system liblz4 via ctypes (argument types declared), or None"""
    try:
        lib = ctypes.CDLL("liblz4.so.1")
    except OSError:
        return None
    sz, vp, szp = ctypes.c_size_t, ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t)
    for name, res, args in (("LZ4F_compressFrameBound", sz, [sz, vp]), ("LZ4F_compressFrame", sz, [vp, sz, ctypes.c_char_p, sz, vp]),
                            ("LZ4F_isError", ctypes.c_uint, [sz]), ("LZ4F_freeDecompressionContext", sz, [vp]),
                            ("LZ4F_createDecompressionContext", sz, [ctypes.POINTER(vp), ctypes.c_uint]),
                            ("LZ4F_decompress", sz, [vp, vp, szp, ctypes.c_char_p, szp, vp])):
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


def liblz4_compress(lib, data: bytes, block_size_id: int = 4, linked: bool = False, block_checksum: bool = False,
                    content_size: bool = False, content_checksum: bool = False, level: int = 0) -> bytes:
    p = _Prefs(blockSizeID=block_size_id, blockMode=0 if linked else 1, contentChecksumFlag=int(content_checksum),
               contentSize=len(data) if content_size else 0, blockChecksumFlag=int(block_checksum), compressionLevel=level)
    cap = lib.LZ4F_compressFrameBound(len(data), ctypes.byref(p))
    out = ctypes.create_string_buffer(cap)
    n = lib.LZ4F_compressFrame(out, cap, data, len(data), ctypes.byref(p))
    if lib.LZ4F_isError(n):
        raise ValueError("LZ4F_compressFrame failed")
    return out.raw[:n]


def liblz4_decompress(lib, frame: bytes, size_hint: int) -> bytes:
    """LZ4F_decompress of one whole frame; raises unless the frame is complete and valid"""
    ctx = ctypes.c_void_p()
    if lib.LZ4F_isError(lib.LZ4F_createDecompressionContext(ctypes.byref(ctx), 100)):
        raise ValueError("no LZ4F context")
    try:
        out = ctypes.create_string_buffer(size_hint + 64)
        dst_n, src_n = ctypes.c_size_t(len(out)), ctypes.c_size_t(len(frame))
        r = lib.LZ4F_decompress(ctx, out, ctypes.byref(dst_n), frame, ctypes.byref(src_n), None)
        if lib.LZ4F_isError(r) or r != 0 or src_n.value != len(frame):
            raise ValueError("LZ4F_decompress rejected the frame")
        return out.raw[:dst_n.value]
    finally:
        lib.LZ4F_freeDecompressionContext(ctx)
