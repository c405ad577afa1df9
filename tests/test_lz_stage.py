"""LZ stage (zstd_lz_kernel's LzSmall / LzBig variants, one CTA per frame, and the pointer-jumping kernels pj_* of
kernels_zstd_pj.cuh): streams written from explicit sequence lists, so that every case lands exactly on one of the
constants where the executors change behaviour, rather than wherever an encoder's match finder happens to put it.

A case is a list of frames, a frame a list of blocks, a block a list of (literal length, match length, offset) sequences
plus its trailing literals.  Every case is pinned twice on the CPU: by execute(), a plain Python LZ executor (the
reference), and by libzstd's (or zlib's) own decode.  zstd streams are written by libzstd's ZSTD_compressSequences with
explicit block delimiters, once with and once without repeat-code resolution; deflate streams by a small fixed-Huffman
writer (RFC 1951 3.2.6).

Constants aimed at (kernels_zstd_lz.cuh, kernels_zstd_pj.cuh; LzSmall / LzBig):
  KEEP 8192 / 65536, BUF 16 KiB / 128 KiB, STEP 3072 / 8192, T 128 / 512 sequences per step (SEQ_RING = 4T),
  LZ_SEQ_MAX 255, LZ_FAR_MAX 32, LIT_RING 4096 / 16384, 16-byte groups, 512-byte flush rows, the pending head group of
  a frame that starts inside a 16-byte group, SEQ_ESC (lengths >= 0xFFFF), PJ_SEG_BLOCKS 1024, PJ_CHASE_HOPS 6,
  32-sequence chunks and 512-byte slices of pj_expand.
"""
import ctypes as C
import os
import random
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

KEEP = {"small": 8192, "big": 65536}
BUF = {"small": 16384, "big": 131072}
STEP = {"small": 3072, "big": 8192}
T = {"small": 128, "big": 512}
LIT_RING = {"small": 4096, "big": 16384}
BLOCK_MAX = 128 * 1024
PJ_SEG_BLOCKS = 1024
ZSTD, DEFLATE = 2, 1


# ---------------------------------------------------------------------------------------------------------------------
# literals and the reference executor

class Lits:
    """Literal bytes of a case: a seeded stream over a 64-symbol alphabet (Huffman-compressible, so that literal-heavy
    blocks still come out as compressed blocks)."""
    _pool = None

    def __init__(self, seed: int):
        if Lits._pool is None:
            Lits._pool = np.random.default_rng(20261022).integers(0, 64, 1 << 20, dtype=np.uint8).tobytes()
        self.p = (seed * 7919) % (1 << 20)

    def take(self, n: int) -> bytes:
        out = []
        while n:
            k = min(n, (1 << 20) - self.p)
            out.append(Lits._pool[self.p:self.p + k])
            self.p = (self.p + k) % (1 << 20)
            n -= k
        return b"".join(out)


def execute(frames, lits: Lits):
    """Run a case's sequences.  Returns (plaintext, valid); a match whose source lies in front of its frame makes the
    case invalid and produces zero bytes in its place (the writer reads literals only)."""
    out = bytearray()
    valid = True
    for fr in frames:
        f0 = len(out)
        for seqs, trail in fr:
            for ll, ml, off in seqs:
                out += lits.take(ll)
                if not ml:
                    continue
                if off == 0 or off > len(out) - f0:
                    valid = False
                    out += bytes(ml)
                    continue
                s = len(out) - off
                if off >= ml:
                    out += out[s:s + ml]
                else:
                    pat = bytes(out[s:])
                    out += (pat * (ml // off + 1))[:ml]
            out += lits.take(trail)
    return bytes(out), valid


# ---------------------------------------------------------------------------------------------------------------------
# zstd writer: libzstd's ZSTD_compressSequences with explicit block delimiters

class _ZSeq(C.Structure):
    _fields_ = [("offset", C.c_uint), ("litLength", C.c_uint), ("matchLength", C.c_uint), ("rep", C.c_uint)]


_ZLIB = None


def _libzstd():
    global _ZLIB
    if _ZLIB is None:
        path = os.environ.get("PNA_ORACLE_LIBZSTD")
        if not path:
            pytest.skip("PNA_ORACLE_LIBZSTD is not set: no libzstd 1.5.7 to write the cases with")
        z = C.CDLL(path)
        if not hasattr(z, "ZSTD_compressSequences"):
            pytest.skip(f"{path} does not export ZSTD_compressSequences")
        z.ZSTD_createCCtx.restype = C.c_void_p
        z.ZSTD_freeCCtx.argtypes = [C.c_void_p]
        z.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
        z.ZSTD_CCtx_setParameter.restype = C.c_size_t
        z.ZSTD_compressSequences.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        z.ZSTD_compressSequences.restype = C.c_size_t
        z.ZSTD_compressBound.argtypes = [C.c_size_t]
        z.ZSTD_compressBound.restype = C.c_size_t
        z.ZSTD_isError.argtypes = [C.c_size_t]
        z.ZSTD_isError.restype = C.c_uint
        z.ZSTD_getErrorName.argtypes = [C.c_size_t]
        z.ZSTD_getErrorName.restype = C.c_char_p
        _ZLIB = z
    return _ZLIB


def zstd_frame(blocks, src: bytes, rep: bool, validate: bool) -> bytes:
    """One frame whose blocks are exactly `blocks` (a delimiter {0, trail, 0} ends each).  rep: the writer turns offsets
    that equal an entry of the repeat history into repeat codes.  validate off lets invalid offsets through."""
    z = _libzstd()
    seqs = []
    for bs, trail in blocks:
        assert sum(ll + ml for ll, ml, _ in bs) + trail <= BLOCK_MAX and (bs or trail)
        seqs += [(off, ll, ml, 0) for ll, ml, off in bs] + [(0, trail, 0, 0)]
    arr = (_ZSeq * len(seqs))(*seqs)
    cc = z.ZSTD_createCCtx()
    try:
        for p, v in ((100, 3),                       # ZSTD_c_compressionLevel
                     (105, 3),                       # ZSTD_c_minMatch: matches of 3 and 4 bytes
                     (1008, 1),                      # ZSTD_c_blockDelimiters: explicit
                     (1009, 1 if validate else 0),   # ZSTD_c_validateSequences
                     (1016, 1 if rep else 2)):       # ZSTD_c_repcodeResolution: enable / disable
            r = z.ZSTD_CCtx_setParameter(cc, p, v)
            assert not z.ZSTD_isError(r), (p, z.ZSTD_getErrorName(r))
        cap = z.ZSTD_compressBound(len(src)) + 1024
        out = C.create_string_buffer(cap)
        n = z.ZSTD_compressSequences(cc, out, cap, arr, len(seqs), src, len(src))
        assert not z.ZSTD_isError(n), z.ZSTD_getErrorName(n)
        return out.raw[:n]
    finally:
        z.ZSTD_freeCCtx(cc)


def zstd_block_types(stream: bytes):
    """Block types (0 raw, 1 RLE, 2 compressed) of every frame of a stream, from the 3-byte block headers."""
    frames, p = [], 0
    while p < len(stream):
        assert int.from_bytes(stream[p:p + 4], "little") == 0xFD2FB528
        fhd = stream[p + 4]
        single = (fhd >> 5) & 1
        p += 5 + (0 if single else 1) + (0, 1, 2, 4)[fhd & 3] + ((1 if single else 0), 2, 4, 8)[fhd >> 6]
        types = []
        while True:
            h = int.from_bytes(stream[p:p + 3], "little")
            last, ty, size = h & 1, (h >> 1) & 3, h >> 3
            types.append(ty)
            p += 3 + (1 if ty == 1 else size)
            if last:
                break
        p += 4 if (fhd >> 2) & 1 else 0
        frames.append(types)
    return frames


# ---------------------------------------------------------------------------------------------------------------------
# deflate writer: fixed Huffman and stored blocks, zlib wrapped

_LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
_LEXT = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
          6145, 8193, 12289, 16385, 24577]
_DEXT = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]


class _Bits:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v: int, n: int):               # LSB first (extra bits, headers)
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def code(self, c: int, n: int):              # Huffman codes go MSB first
        self.put(int(format(c, f"0{n}b")[::-1], 2), n)

    def align(self):
        if self.n:
            self.put(0, 8 - self.n)


def _fixed_sym(w: _Bits, s: int):
    if s < 144:
        w.code(0x30 + s, 8)
    elif s < 256:
        w.code(0x190 + s - 144, 9)
    elif s < 280:
        w.code(s - 256, 7)
    else:
        w.code(0xC0 + s - 280, 8)


def deflate_stream(blocks, lits: Lits):
    """blocks: ("fixed", tokens) or ("stored", n).  Tokens: ("lit", n), ("match", length, dist), ("lsym", 286 | 287),
    ("dsym", 30 | 31).  Returns (zlib stream, plaintext, valid)."""
    w = _Bits()
    w.out += b"\x78\x01"
    out = bytearray()
    valid = True
    for bi, (kind, body) in enumerate(blocks):
        final = 1 if bi == len(blocks) - 1 else 0
        if kind == "stored":
            w.put(final, 1)
            w.put(0, 2)
            w.align()
            data = lits.take(body)
            w.put(len(data), 16)
            w.put(len(data) ^ 0xFFFF, 16)
            w.out += data
            out += data
            continue
        w.put(final, 1)
        w.put(1, 2)
        for t in body:
            if t[0] == "lit":
                data = lits.take(t[1])
                for b in data:
                    _fixed_sym(w, b)
                out += data
            elif t[0] == "match":
                _, ln, d = t
                assert 3 <= ln <= 258 and 1 <= d <= 32768
                lc = max(k for k in range(29) if _LBASE[k] <= ln) if ln < 258 else 28
                _fixed_sym(w, 257 + lc)
                w.put(ln - _LBASE[lc], _LEXT[lc])
                dc = max(k for k in range(30) if _DBASE[k] <= d)
                w.code(dc, 5)
                w.put(d - _DBASE[dc], _DEXT[dc])
                if d > len(out):
                    valid = False
                    out += bytes(ln)
                else:
                    s = len(out) - d
                    out += bytes(out[s:s + ln]) if d >= ln else (bytes(out[s:]) * (ln // d + 1))[:ln]
            elif t[0] == "lsym":
                _fixed_sym(w, t[1])
                w.put(0, 16)
                valid = False
            elif t[0] == "dsym":
                _fixed_sym(w, 257)
                w.code(t[1], 5)
                w.put(0, 16)
                valid = False
        _fixed_sym(w, 256)
    w.align()
    w.out += zlib.adler32(bytes(out)).to_bytes(4, "big")
    return bytes(w.out), bytes(out), valid


# ---------------------------------------------------------------------------------------------------------------------
# the cases

ALL = ("small", "big", "pj")


class Case:
    def __init__(self, name, kind, stream, plain, err=None, execs=ALL, slow=False, compressed=None, cap=None):
        self.name, self.kind, self.stream, self.plain, self.err = name, kind, stream, plain, err
        self.execs, self.slow, self.compressed = execs, slow, compressed
        self.cap = cap                    # output capacity of the decode with a size hint (None: exactly len(plain))


def chop(seqs, per_block, trail_last=0):
    """Cut a sequence list into blocks of per_block sequences (fewer where BLOCK_MAX would be exceeded)."""
    blocks, cur, size = [], [], 0
    for s in seqs:
        n = s[0] + s[1]
        if cur and (len(cur) == per_block or size + n > BLOCK_MAX):
            blocks.append((cur, 0))
            cur, size = [], 0
        cur.append(s)
        size += n
    blocks.append((cur, trail_last))
    return blocks


def lit_blocks(n):
    """n literal bytes as all-literal blocks."""
    return [([], min(BLOCK_MAX, n - k)) for k in range(0, n, BLOCK_MAX)]


def zstd_case(name, frames, seed, rep, slow=False, err=None, execs=ALL):
    """Execute and write one zstd case.  Blocks of >= 32 bytes that are at least half match bytes must come out
    compressed (checked by test_lz_cases_pinned)."""
    plain, valid = execute(frames, Lits(seed))
    assert valid == (err is None), name
    stream, pos = b"", 0
    need = []
    for fr in frames:
        n = sum(sum(ll + ml for ll, ml, _ in bs) + t for bs, t in fr)
        stream += zstd_frame(fr, plain[pos:pos + n], rep, validate=err is None)
        pos += n
        need.append([sum(ml for _, ml, _ in bs) * 2 >= sum(ll + ml for ll, ml, _ in bs) + t
                     and sum(ll + ml for ll, ml, _ in bs) + t >= 32 for bs, t in fr])
    return Case(f"{name}_r{int(rep)}", ZSTD, stream, None if err else plain, err=err, execs=execs, slow=slow, compressed=need)


def _window_edge(v, rnd):
    """Offsets KEEP-1 .. KEEP+17 x lengths 3 .. 256, each match start at all 16 phases mod 16, in a frame longer than
    BUF (so that some land right after a window slide)."""
    keep = KEEP[v]
    seqs, pos = [], keep + 700
    for rnd_pass in range(2):
        for off in (keep - 1, keep, keep + 1, keep + 15, keep + 16, keep + 17):
            for ml in (3, 4, 31, 32, 33, 255, 256):
                for ph in rnd.sample(range(16), 16):
                    ll = 1 + (ph - (pos + 1)) % 16 + 16 * rnd_pass
                    seqs.append((ll, ml, off))
                    pos += ll + ml
    assert pos > BUF[v]
    return [lit_blocks(keep + 700) + chop(seqs, 48, trail_last=5)]


def _far_sweep(v, rnd):
    """Every offset KEEP-64 .. KEEP+600 over a ~300 KiB frame: far sources fetched one step ahead, against the 512-byte
    flush mark."""
    keep = KEEP[v]
    seqs, pos = [], keep + 600
    while pos < 300 << 10:
        for off in range(keep - 64, keep + 601):
            ll, ml = rnd.randrange(1, 25), rnd.choice((3, 4, 7, 16, 17, 31, 32, 33, 40))
            seqs.append((ll, ml, off))
            pos += ll + ml
    return [lit_blocks(keep + 600) + chop(seqs, 700)]


def _overlap(rnd):
    """Offsets 1..20 and 31..33 under lengths up to 255 (periodic codes) and 256..1000 (whole-CTA copies)."""
    seqs = []
    for off in list(range(1, 21)) + [31, 32, 33]:
        for ml in (3, 4, 5, off, off + 1, 2 * off, 2 * off + 1, 31, 32, 33, 100, 254, 255, 256, 257, 300, 511, 512, 777, 1000):
            if ml >= 3:
                seqs.append((rnd.randrange(0, 3), ml, off))
    # chains: each match's source is the previous match, all inside one step
    for _ in range(60):
        prev = rnd.randrange(8, 40)
        seqs.append((rnd.randrange(1, 4), prev, rnd.randrange(1, 9)))
        for _ in range(rnd.randrange(3, 8)):
            ml = rnd.randrange(3, 60)
            seqs.append((0, ml, prev - rnd.randrange(0, min(prev, 4))))
            prev = ml
    return [[([], 64)] + chop(seqs, 64, trail_last=3)]


def _step_groups(v, rnd, d):
    """Blocks whose sequences reach STEP + d bytes exactly at a sequence end, three times over."""
    seqs, pos = [], 2048
    for _ in range(3):
        rem = STEP[v] + d
        while rem:
            if rem > 80:
                ll, ml = rnd.randrange(0, 11), rnd.randrange(3, 61)
            else:
                ll = rem // 3
                ml = rem - ll
            off = rnd.choice((rnd.randrange(1, 40), rnd.randrange(1, min(pos, 2000)), pos - rnd.randrange(0, 16)))
            seqs.append((ll, ml, max(1, min(off, pos + ll))))
            pos += ll + ml
            rem -= ll + ml
    return seqs


def _step_cut(v, rnd):
    """Step cuts at STEP - 1, STEP, STEP + 1 bytes; blocks of T - 1, T, T + 1, 4T (SEQ_RING) and 4T + 1 sequences."""
    blocks = [([], 2048)]
    for d in (-1, 0, 1):
        blocks.append((_step_groups(v, rnd, d), 0))
    for n in (T[v] - 1, T[v], T[v] + 1, 4 * T[v], 4 * T[v] + 1):
        blocks.append(([(rnd.randrange(0, 3), rnd.randrange(3, 7), rnd.randrange(1, 300)) for _ in range(n)], rnd.randrange(0, 3)))
    return [blocks]


def _long_short(rnd):
    """255 / 256 lengths first, last and in pairs; literal runs at LIT_RING -1/0/+1; trailing literals 0..4096."""
    blocks = [([], 20000)]
    small = lambda k: [(rnd.randrange(0, 4), rnd.randrange(3, 20), rnd.randrange(1, 5000)) for _ in range(k)]
    for L in (254, 255, 256, 257):
        blocks.append(([(L, 20, 7)] + small(5), 1))
        blocks.append(([(0, L, 5000)] + small(5), 0))
        blocks.append(([(0, L, 3)] + small(3) + [(2, L, 11)], 0))
        blocks.append((small(4) + [(1, L, 9), (0, L, 4000), (L, L, 40)], 2))
    for lr in (4096, 16384):
        for n in (lr - 1, lr, lr + 1):
            blocks.append((small(3) + [(n, 8, 3)] + small(3) + [(n, 300, 1000)], 0))
    for t in (0, 1, 15, 16, 4096):
        blocks.append((small(6), t))
    return [blocks]


def _long_esc(rnd):
    """Escape records: lengths 65534..65536 and ~131000, first, last and two in a row."""
    blocks = lit_blocks(70000)
    for L in (65534, 65535, 65536):
        blocks.append(([(L, 20, 7), (0, 30, 70000)], 3))
        blocks.append(([(0, L, 70000), (2, 40, 5)], 0))
        blocks.append(([(5, 10, 3), (1, L, 13)], 0))
        blocks.append(([(0, L, 1), (0, L, 69999 - (L & 7))] if 2 * L <= BLOCK_MAX else [(0, L, 1), (0, BLOCK_MAX - L, 4)], 0))
        blocks.append(([(L, L - 1, 65536 + 5)], 1))
    blocks.append(([(131000, 40, 100000)], 4))
    blocks.append(([(3, 131000, 70000)], 0))
    blocks.append(([(0, 131000, 2), (1, 20, 9)], 0))
    return [blocks]


def _block_structure(rnd):
    """Many tiny blocks whose matches reach into earlier blocks; > 32 blocks carrying a repeat history."""
    blocks, pos = [([], 200)], 200
    for _ in range(400):
        size = rnd.randrange(1, 65)
        if size < 4:
            blocks.append(([], size))
        else:
            ml = rnd.randrange(3, size + 1)
            ll = rnd.randrange(0, size - ml + 1)
            blocks.append(([(ll, ml, rnd.randrange(ll + 1, pos + ll + 1))], size - ll - ml))
        pos += size
    offs = (17, 40, 333, 1000)
    for _ in range(80):
        bs = []
        for _ in range(6):
            off = rnd.choice(offs) if rnd.random() < 0.8 else rnd.randrange(1, 3000)
            bs.append((rnd.choice((0, 0, 1, 3)), rnd.randrange(3, 40), off))
        blocks.append((bs, rnd.randrange(0, 3)))
    return [blocks]


def _frame_body(v, rnd, n):
    """A frame of about n bytes: it opens with offsets 1, 4, 8 (the reset repeat history, ll = 0 forms included), then
    near and far matches whose source is byte 0..15 of the frame, then ordinary traffic."""
    seqs = [(1, 5, 1), (0, 6, 4), (0, 7, 8), (2, 4, 1), (0, 5, 8), (0, 3, 4), (1, 9, 4), (0, 4, 1)]
    pos = sum(ll + ml for ll, ml, _ in seqs)
    while pos < n - 64:
        if rnd.random() < 0.35:
            j = rnd.randrange(16)
            ll = rnd.randrange(0, 8)
            ml = rnd.choice((3, 8, 16, 17, 32, 40, 300))
            seqs.append((ll, ml, pos + ll - j))
        else:
            ll, ml = rnd.randrange(0, 30), rnd.randrange(3, 80)
            seqs.append((ll, ml, rnd.randrange(1, pos + ll + 1)))
        pos += seqs[-1][0] + seqs[-1][1]
    blocks = chop(seqs, 100)
    return blocks, pos


def _multi_frame(v, rnd, counts):
    """Streams of 2..5 frames; the frame starts take every output phase mod 16 once.  Frames after the first are longer
    than KEEP.  Returns a list of frame lists."""
    streams, phase = [], 0
    for cnt in counts:
        frames, at = [], 0
        for k in range(cnt):
            blocks, n = _frame_body(v, rnd, KEEP[v] + rnd.randrange(500, 2500) if k else rnd.randrange(200, 3000))
            if k + 1 < cnt:   # pad with trailing literals so that the next frame starts at the next phase
                pad = (phase - (at + n)) % 16
                blocks[-1] = (blocks[-1][0], blocks[-1][1] + pad)
                n += pad
                phase = (phase + 1) % 16
            frames.append(blocks)
            at += n
        streams.append(frames)
    return streams


def _pj_segments(rnd, nblk, lo, hi):
    """nblk blocks of lo..hi bytes (several pointer-jumping segments); sources up to a few blocks back, so pointers leave
    their segment at every segment start."""
    blocks, pos = [([], 4096)], 4096
    for _ in range(nblk):
        size = rnd.randrange(lo, hi)
        bs, got = [], 0
        while got < size - 40:
            ll, ml = rnd.randrange(0, 6), rnd.randrange(8, 120)
            bs.append((ll, ml, rnd.randrange(max(1, ll + 1), min(pos + got + ll, 4 * hi) + 1)))
            got += ll + ml
        blocks.append((bs, 2))
        pos += got + 2
    return [blocks]


def _pj_chains(rnd, total):
    """A 1 KiB seed copied forward at offset 1024 (chains of total / 1024 hops), then an offset-1 run across many
    blocks (four sequences per block, so that the writer keeps them as compressed blocks)."""
    blocks = [([], 1024)]
    for _ in range(total // 16384):
        blocks.append(([(0, 4096, 1024)] * 4, 0))
    blocks.append(([(1, 50, 1)] + [(0, 50, 1)] * 3, 0))
    for _ in range(40):
        blocks.append(([(0, 200, 1)] * 4, 0))
    blocks.append(([(0, 10, 1)], 1))
    return [blocks]


def _pj_shapes(rnd):
    """Blocks of 31, 32 and 33 sequences (pj_expand's 32-sequence chunks); literal runs and matches that span many of
    pj_expand's 512-byte slices."""
    blocks, pos = [([], 8192)], 8192
    for n in (31, 32, 33, 63, 64, 65):
        bs = [(rnd.randrange(0, 5), rnd.randrange(3, 50), rnd.randrange(1, 8000)) for _ in range(n)]
        blocks.append((bs, rnd.randrange(0, 2)))
    blocks.append(([(5000, 5000, 3000), (20000, 30000, 7), (1, 7000, 8000)], 600))
    blocks.append(([(0, 9000, 511), (0, 2049, 513), (3, 60000, 20000)], 0))
    return [blocks]


def _invalid(v, where, far, long_):
    """A match at frame position p whose offset is p + 1: in the first block, in a later block (one byte in front of the
    frame) or in the second frame of a stream (the last byte of the first frame)."""
    ml = 300 if long_ else 10
    seqs, pos = [], 0
    while pos < (KEEP[v] + 200 if far else 100):   # literal chunks below 0xFFFF: only the bad match takes the long path
        seqs.append((min(30000, (KEEP[v] + 200 if far else 100) - pos), 10, 5))
        pos += seqs[-1][0] + 10
    ok = [(3, 20, 2), (0, 12, 30), (4, 8, 17)]
    if where == "first":
        return [[(seqs + [(3, ml, pos + 3 + 1)] + ok, 2)]]
    if where == "block":
        return [[(seqs, 3), ([(3, ml, pos + 3 + 3 + 1)] + ok, 1)]]
    return [[([(700, 20, 300)], 5)], [(seqs + [(3, ml, pos + 3 + 1)] + ok, 2)]]


def _deflate_cases(rnd):
    out = []
    lens = [("match", L, rnd.choice((1, 2, 3, 7, 100, 258, 300))) for L in range(3, 259)]
    toks = [("lit", 300)] + [t for L in lens for t in (L, ("lit", rnd.randrange(0, 3)))]
    out.append(("df_lengths", [("fixed", toks)]))
    far = [("lit", 33000)]
    for d in (1, 8191, 8192, 8193, 32768):
        for L in (3, 32, 33, 255, 258):
            far += [("match", L, d), ("lit", rnd.randrange(0, 5))]
    out.append(("df_distances", [("fixed", far)]))
    out.append(("df_dist_eq_produced", [("fixed", [("lit", 777), ("match", 40, 777), ("lit", 3), ("match", 258, 820)])]))
    runs = [("lit", 10)]
    for n in (65534, 65535, 65536):
        runs += [("match", 20, 7), ("lit", n), ("match", 258, 30000), ("match", 3, 32768)]
    out.append(("df_literal_runs", [("fixed", runs)]))
    out.append(("df_blocks", [("fixed", [("lit", 500), ("match", 100, 300)]), ("stored", 3000),
                              ("fixed", [("match", 258, 3200), ("lit", 4), ("match", 30, 1)]), ("stored", 0),
                              ("fixed", [("match", 12, 3800)])]))
    bad = [("df_bad_dist_gt_produced", [("fixed", [("lit", 777), ("match", 40, 778)])]),
           ("df_bad_dist_gt_produced_later", [("fixed", [("lit", 500)]), ("stored", 500),
                                              ("fixed", [("match", 10, 100), ("match", 258, 1111)])])]
    for s in (30, 31):
        bad.append((f"df_bad_dsym{s}", [("fixed", [("lit", 100), ("dsym", s), ("lit", 10)])]))
    for s in (286, 287):
        bad.append((f"df_bad_lsym{s}", [("fixed", [("lit", 100), ("lsym", s), ("lit", 10)])]))
    cases = []
    for name, blocks in out + bad:
        stream, plain, valid = deflate_stream(blocks, Lits(len(cases) + 5000))
        assert valid == (not name.startswith("df_bad")), name
        cases.append(Case(name, DEFLATE, stream, plain if valid else None, err=None if valid else "input", execs=("small", "big")))
    return cases


def cases():
    """Every case, deterministic.  Names say the family, the constant aimed at and _r0 / _r1 (without / with repeat
    codes)."""
    out = []
    rnd = random.Random(1022)
    seed = iter(range(1, 10 ** 6))
    for rep in (False, True):
        for v in ("small", "big"):
            out.append(zstd_case(f"window_edge_{v}", _window_edge(v, rnd), next(seed), rep))
            out.append(zstd_case(f"far_sweep_{v}", _far_sweep(v, rnd), next(seed), rep))
            out.append(zstd_case(f"step_cut_{v}", _step_cut(v, rnd), next(seed), rep))
            for i, frames in enumerate(_multi_frame(v, rnd, (2, 3, 4, 5, 5, 3) if v == "small" else (5, 5, 5, 5))):
                out.append(zstd_case(f"multi_frame_{v}{i}", frames, next(seed), rep, slow=v == "big"))
            for where in ("first", "block", "frame"):
                for far in (False, True):
                    for long_ in (False, True):
                        out.append(zstd_case(f"bad_offset_{v}_{where}_{'far' if far else 'near'}_{'long' if long_ else 'short'}",
                                             _invalid(v, where, far, long_), next(seed), rep, err="data"))
        out.append(zstd_case("overlap", _overlap(rnd), next(seed), rep))
        out.append(zstd_case("long_short", _long_short(rnd), next(seed), rep))
        out.append(zstd_case("long_esc", _long_esc(rnd), next(seed), rep, slow=True))
        out.append(zstd_case("block_structure", _block_structure(rnd), next(seed), rep))
        out.append(zstd_case("pj_segments", _pj_segments(rnd, PJ_SEG_BLOCKS + 76, 100, 300), next(seed), rep))
        out.append(zstd_case("pj_segments_large", _pj_segments(rnd, 2500, 1024, 2048), next(seed), rep, slow=True))
        out.append(zstd_case("pj_chains", _pj_chains(rnd, 64 << 10), next(seed), rep))
        out.append(zstd_case("pj_chains_large", _pj_chains(rnd, 2 << 20), next(seed), rep, slow=True))
        out.append(zstd_case("pj_shapes", _pj_shapes(rnd), next(seed), rep))
    # capacity: one entry of many blocks and one of a few, each decoded into one byte less than it needs
    for c in list(out):
        if c.name in ("pj_segments_r1", "overlap_r1"):
            out.append(Case(c.name + "_cap", ZSTD, c.stream, c.plain, err="nospace", compressed=c.compressed, cap=len(c.plain) - 1))
    out += _deflate_cases(rnd)
    return out


@pytest.fixture(scope="module")
def lz_cases():
    return cases()


# ---------------------------------------------------------------------------------------------------------------------
# tests

def test_lz_cases_pinned(oracle, lz_cases):
    names = [c.name for c in lz_cases]
    assert len(names) == len(set(names))
    for c in lz_cases:
        if c.kind == ZSTD:
            types = zstd_block_types(c.stream)
            assert [len(t) for t in types] == [len(n) for n in c.compressed], c.name   # the writer kept every block
            for ft, fn in zip(types, c.compressed):
                assert all(t == 2 for t, n in zip(ft, fn) if n), (c.name, ft)
            if c.plain is None:
                with pytest.raises(oracle.OracleError):
                    oracle.decompress(ZSTD, c.stream, 1 << 20)
            else:
                assert oracle.decompress(ZSTD, c.stream, len(c.plain)) == c.plain, c.name
        elif c.plain is None:
            with pytest.raises(zlib.error):
                zlib.decompress(c.stream)
        else:
            assert zlib.decompress(c.stream) == c.plain, c.name


@pytest.fixture(scope="module")
def hc(built):
    L = C.CDLL(os.path.join(HERE, "host", "libpna_hostcore.so"))
    L.hc_zstd_decode.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p]
    L.hc_inflate.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    return L


def test_lz_cases_host_core(hc, lz_cases):
    for c in lz_cases:
        if c.err == "nospace":
            continue
        cap = (len(c.plain) if c.plain is not None else 0) + (64 << 10) + (4 << 20) * (c.plain is None)
        out = C.create_string_buffer(cap)
        n = C.c_uint64(0)
        if c.kind == ZSTD:
            st = hc.hc_zstd_decode(c.stream, len(c.stream), out, cap, C.byref(n), None)
        else:
            st = hc.hc_inflate(c.stream, len(c.stream), out, cap, C.byref(n))
        if c.err:
            assert st != 0, f"{c.name}: accepted"
        else:
            assert st == 0 and out.raw[:n.value] == c.plain, (c.name, st)


# PNA_LZ_PJ_MIN_BLOCKS=0 turns pointer jumping off, =1 sends every zstd entry to it; PNA_LZ_VARIANT forces the CTA variant
EXECUTORS = {"small": {"PNA_LZ_VARIANT": "s", "PNA_LZ_PJ_MIN_BLOCKS": "0"},
             "big": {"PNA_LZ_VARIANT": "b", "PNA_LZ_PJ_MIN_BLOCKS": "0"},
             "pj": {"PNA_LZ_VARIANT": None, "PNA_LZ_PJ_MIN_BLOCKS": "1"}}


def _run_batch(ctx, pna, batch, hinted):
    """Decode a batch in one call (with exact size hints and capacities, or through the sizing pass) and check every
    entry: status, length and bytes."""
    want = {None: pna.OK, "data": pna.E_INVALID_DATA, "input": pna.E_INVALID_INPUT, "nospace": pna.E_NOSPACE}
    entries, caps = [], []
    for c in batch:
        n = len(c.plain) if c.plain is not None else None
        entries.append({"bodies": [c.stream], "compression": c.kind, "encryption": 0, "cipher_mode": 0, "key": None,
                        "raw_size_hint": n if hinted else None})
        caps.append(c.cap if c.cap is not None else (n if n is not None else 1 << 20))
    outs, st, lens = ctx.decode_batch(entries, caps=caps if hinted else None)
    bad = []
    for c, o, s, n in zip(batch, outs, st, lens):
        exp = want[c.err] if (hinted or c.err != "nospace") else pna.OK   # the sizing pass gives a nospace case its room
        if s != exp:
            bad.append((c.name, "status", int(s), exp))
        elif exp in (pna.OK, pna.E_NOSPACE) and n != len(c.plain):
            bad.append((c.name, "len", int(n), len(c.plain)))
        elif exp == pna.OK and o.tobytes() != c.plain:
            got = o.tobytes()
            first = next((i for i, (a, b) in enumerate(zip(got, c.plain)) if a != b), min(len(got), len(c.plain)))
            bad.append((c.name, "bytes", "first difference at", first))
    assert not bad, (len(bad), bad)


@pytest.mark.gpu
@pytest.mark.parametrize("executor,large", [pytest.param(e, lg, id=e + ("-large" if lg else ""), marks=[pytest.mark.slow_emu] if lg else [])
                                            for lg in (False, True) for e in EXECUTORS])
def test_lz_cases_gpu(ctx, pna, lz_cases, monkeypatch, executor, large):
    for k, val in EXECUTORS[executor].items():
        if val is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, val)
    batch = [c for c in lz_cases if executor in c.execs and c.slow == large]
    for hinted in (True, False):
        _run_batch(ctx, pna, batch, hinted)
    if executor == "pj" and not large:
        # one batch that mixes pointer-jumping entries (>= 40 blocks) with entries the CTA-per-frame kernel takes
        monkeypatch.setenv("PNA_LZ_PJ_MIN_BLOCKS", "40")
        _run_batch(ctx, pna, [c for c in batch if c.kind == ZSTD], True)
