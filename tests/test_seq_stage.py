"""zstd sequence stage (SeqStream, run by zstd_seq_kernel on the GPU and by the host core on the CPU): frames that take
the decode loop's rare paths, each checked against libzstd's decode.

- offsets of 2^23 and more with long literal and match lengths (a window of 2^25 with long-distance matching), the
  sequences of more than 64 bits that need a second bit window
- literal and match lengths of 0xFFFF and more (the escape records)
- repeat offsets, predefined / RLE / repeat table modes, blocks with 0, 1 and many sequences
- every bitstream start phase modulo 16 (a skippable frame of 0..15 bytes in front)
- bit flips in the last bytes of the frame and truncations
"""
import ctypes as C
import os
import random
import struct

import numpy as np
import pytest

import corpus

HERE = os.path.dirname(os.path.abspath(__file__))


def _zstd():
    for name in (os.environ.get("PNA_ORACLE_ZSTD"), "libzstd.so.1", "libzstd.so"):
        if name:
            try:
                z = C.CDLL(name)
                break
            except OSError:
                pass
    else:
        pytest.skip("no libzstd")
    z.ZSTD_createCCtx.restype = C.c_void_p
    z.ZSTD_freeCCtx.argtypes = [C.c_void_p]
    z.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
    z.ZSTD_CCtx_setParameter.restype = C.c_size_t
    z.ZSTD_compress2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    z.ZSTD_compress2.restype = C.c_size_t
    z.ZSTD_compressBound.argtypes = [C.c_size_t]
    z.ZSTD_compressBound.restype = C.c_size_t
    z.ZSTD_isError.argtypes = [C.c_size_t]
    z.ZSTD_isError.restype = C.c_uint
    return z


def compress(data: bytes, level: int, window_log: int = 0, ldm: bool = False) -> bytes:
    z = _zstd()
    cc = z.ZSTD_createCCtx()
    try:
        z.ZSTD_CCtx_setParameter(cc, 100, level)              # ZSTD_c_compressionLevel
        z.ZSTD_CCtx_setParameter(cc, 200, 0)                  # ZSTD_c_contentSizeFlag: a flip must show in the decode,
                                                              # not only against the frame header's size
        if window_log:
            z.ZSTD_CCtx_setParameter(cc, 101, window_log)     # ZSTD_c_windowLog
        if ldm:
            z.ZSTD_CCtx_setParameter(cc, 160, 1)              # ZSTD_c_enableLongDistanceMatching
        cap = z.ZSTD_compressBound(len(data))
        out = C.create_string_buffer(cap)
        n = z.ZSTD_compress2(cc, out, cap, data, len(data))
        assert not z.ZSTD_isError(n)
        return out.raw[:n]
    finally:
        z.ZSTD_freeCCtx(cc)


def _rand(seed: int, n: int) -> bytes:
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def _cases():
    """(name, frame, plain) of valid frames."""
    out = []
    # far offsets (codes 23-24) carrying 16-bit literal and match length extras: 55+ value bits before the states
    a, c = _rand(1, 90000), _rand(3, 70000)
    far = a + _rand(2, 9 << 20) + c + a + c[:40000] + bytes(5000) + a[:70000]
    out.append(("far_long", compress(far, 3, window_log=25, ldm=True), far))
    # lengths >= 0xFFFF: long zero runs (match lengths) and long literal runs in front of a match
    esc = bytes(300000) + _rand(4, 100000) + bytes(200000) + _rand(5, 65535) + b"x" * 65535 + _rand(6, 65534) + bytes(70000)
    out.append(("escapes", compress(esc, 3), esc))
    # repeat offsets: records with a few recurring strides, where the optimal parser uses rep1 / rep2 / rep0 - 1
    rnd = random.Random(7)
    recs = []
    words = [_rand(100 + k, 8) for k in range(6)]
    for i in range(20000):
        w = words[rnd.randrange(6)]
        recs.append(w[: rnd.choice((3, 4, 5, 8))] + bytes([i & 0xFF, rnd.randrange(4)]))
    rep = b"".join(recs)
    for lvl in (1, 9, 19, 22):
        out.append((f"repeats_l{lvl}", compress(rep, lvl), rep))
    # table modes: a handful of sequences (predefined tables), a periodic run whose codes are all equal (RLE tables),
    # many blocks of the same statistics (repeat mode)
    out.append(("predef", compress(b"abcdefgh" * 3 + b"zz" + b"abcdefgh" * 2, 3), b"abcdefgh" * 3 + b"zz" + b"abcdefgh" * 2))
    per = (b"0123456789abcdef" * 4 + _rand(8, 3)) * 3000
    out.append(("rle_codes", compress(per, 3), per))
    many = corpus.make_file(11, 1 << 20)
    out.append(("repeat_mode", compress(many, 5), many))
    # 0 sequences (all literals), 1 sequence, and one block of many short sequences
    out.append(("zero_seq", compress(_rand(9, 20000), 3), _rand(9, 20000)))
    one = _rand(10, 500) + _rand(10, 500)
    out.append(("one_seq", compress(one, 3), one))
    short = bytes(rnd.randrange(4) for _ in range(120000))
    out.append(("many_seq", compress(short, 19), short))
    # every start phase of the stream modulo 16: a skippable frame of k bytes in front
    base = corpus.make_file(12, 60000)
    fb = compress(base, 3)
    for k in range(16):
        skip = struct.pack("<II", 0x184D2A50, k) + bytes(k) if k else b""
        out.append((f"phase{k}", skip + fb, base))
    return out


@pytest.fixture(scope="module")
def cases():
    return _cases()


def _corrupt(cases):
    """Bit flips in the last 16 bytes and truncations of a few frames: the sequence bitstream is the end of a block."""
    rnd = random.Random(13)
    out = []
    for name, f, plain in cases:
        if not name.startswith(("far_long", "escapes", "repeats_l19", "rle_codes", "phase3")):
            continue
        for _ in range(24):
            b = bytearray(f)
            b[len(b) - 1 - rnd.randrange(16)] ^= 1 << rnd.randrange(8)
            out.append((name + "_flip", bytes(b), len(plain)))
        for cut in (1, 2, 3, 5, 9):
            out.append((name + "_cut", f[:-cut], len(plain)))
    return out


def _libzstd(oracle, frame, cap):
    try:
        return 0, oracle.decompress(2, frame, cap + 4096)
    except oracle.OracleError:
        return 1, None


def _hc_decode(hc, frame, cap):
    out = C.create_string_buffer(cap + 4096)
    n = C.c_uint64(0)
    st = hc.hc_zstd_decode(frame, len(frame), out, cap + 4096, C.byref(n), None)
    return st, (out.raw[:n.value] if st == 0 else None)


@pytest.fixture(scope="module")
def hc(built):
    L = C.CDLL(os.path.join(HERE, "host", "libpna_hostcore.so"))
    L.hc_zstd_decode.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p]
    return L


def test_seq_stage_host_core(hc, oracle, cases):
    for name, f, plain in cases:
        assert oracle.decompress(2, f, len(plain)) == plain, name
        st, o = _hc_decode(hc, f, len(plain))
        assert st == 0 and o == plain, name
    for name, f, cap in _corrupt(cases):
        rst, ref = _libzstd(oracle, f, cap)
        st, o = _hc_decode(hc, f, cap)
        if rst == 0 and st == 0:
            assert o == ref, name
        elif rst != 0:
            assert st != 0, f"{name}: accepted what libzstd rejects"
        else:   # the one documented class: a Huffman literal stream that over-reads (test_host_cores.py)
            assert hc.hc_site_value() == 10, f"{name}: rejected what libzstd accepts"


@pytest.mark.gpu
def test_seq_stage_gpu(ctx, hc, cases):
    frames = [(n, f, len(p)) for n, f, p in cases] + _corrupt(cases)
    entries = [{"bodies": [f], "compression": 2, "encryption": 0, "cipher_mode": 0, "key": None, "raw_size_hint": cap}
               for _, f, cap in frames]
    outs, st, lens = ctx.decode_batch(entries, caps=[cap + 4096 for _, _, cap in frames])
    for (name, f, cap), o, s, n in zip(frames, outs, st, lens):
        hst, ho = _hc_decode(hc, f, cap)
        assert (s == 0) == (hst == 0), (name, s, hst)
        if s == 0:
            assert o[:n].tobytes() == ho, name
