"""AES-256-CTR tile kernels (extract: aes_ctr_tiles_kernel, create: encrypt_tiles_kernel) and the counter-run cache
(aes256_ctr_run_init / aes256_ctr_run_block) byte for byte against OpenSSL through the oracle.

Extract tiles are cut at body boundaries and after 32 counter runs of 256 blocks (8192 blocks); the cases below put
run starts, tile ends, body boundaries and the 2^128 counter wrap where the kernel has to get them right."""
import ctypes as C
import os
import random
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CORE = os.path.join(os.path.dirname(HERE), "portable-network-archive_b200", "csrc", "cipher_core.cuh")

TILE_BLOCKS = 32 * 256


def _iv(low: bytes, rnd: random.Random) -> bytes:
    return bytes(rnd.randrange(256) for _ in range(16 - len(low))) + low


IV_CLASSES = [b"\x00", b"\x01", b"\xfe", b"\xff", b"\xff" * 4, b"\xff" * 8, b"\xff" * 16, b"\xff" * 15 + b"\x00",
              b"\xff\xff\xff\xfe\xff\xff\xff\xff"]


# ---------------------------------------------------------------------------------------------------- CPU tier
_SHIM = r"""
#include "%s"
using namespace pna;
extern "C" void run_keystream(const uint8_t* key, const uint8_t* ivb, uint64_t first, uint64_t n, uint8_t* out) {
    static AesTables T; static bool init = false;
    if (!init) { aes_make_tables(&T); init = true; }
    AesKey K; aes256_expand_key(&T, key, &K);
    const Te0Rot t{T.te0};
    uint32_t iv[4]; memcpy(iv, ivb, 16);
    uint32_t p[5], run[4];
    bool have = false;
    for (uint64_t b = first; b < first + n; b++) {
        uint32_t c[4]; ctr128be_add(iv, b, c);
        if (!have || (c[3] >> 24) == 0) {   // a new counter run
            memcpy(run, c, 16); run[3] &= 0x00FFFFFFu;
            aes256_ctr_run_init(run, K.rk, t, p);
            have = true;
        }
        uint32_t s[4]; aes256_ctr_run_block(p, c[3] & 0xFF000000u, K.rk, t, s);
        uint32_t r[4]; memcpy(r, c, 16); aes256_encrypt_block4(r, K.rk, t);
        if (memcmp(r, s, 16)) memset(s, 0, 16);   // the plain four-table block must agree
        memcpy(out + 16 * (b - first), s, 16);
    }
}
"""


@pytest.fixture(scope="module")
def run_core(tmp_path_factory):
    d = tmp_path_factory.mktemp("ctr_core")
    src, so = d / "shim.cpp", d / "libctr.so"
    src.write_text(_SHIM % CORE)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", str(so), str(src)])
    L = C.CDLL(str(so))
    L.run_keystream.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_char_p]
    return L


@pytest.mark.parametrize("low", IV_CLASSES, ids=lambda b: b.hex())
def test_counter_run_core_matches_openssl(run_core, oracle, low):
    rnd = random.Random(low)
    key, iv = os.urandom(32), _iv(low, rnd)
    for first, n in [(0, 1), (0, 300), (3, 600), (250, 10), (255, 2), (256, 257), (1000, 40)]:
        out = C.create_string_buffer(16 * n)
        run_core.run_keystream(key, iv, first, n, out)
        want = oracle.ctr(1, key, iv, bytes(16 * (first + n)))[16 * first:]
        assert out.raw == want, (iv.hex(), first, n)


# ---------------------------------------------------------------------------------------------------- GPU tier
def _stream(oracle, plain, key, iv):
    return oracle.encode_stream(plain, 0, -1, 1, 1, key, iv)


def _decode(ctx, streams, keys, cuts=None):
    entries = []
    for i, (s, k) in enumerate(zip(streams, keys)):
        bounds = [0] + sorted(set(c for c in (cuts[i] if cuts else []) if 0 < c < len(s))) + [len(s)]
        entries.append({"bodies": [s[a:b] for a, b in zip(bounds, bounds[1:])], "compression": 0, "encryption": 1,
                        "cipher_mode": 1, "key": k, "raw_size_hint": max(len(s) - 16, 0)})
    outs, st, _ = ctx.decode_batch(entries, caps=[max(len(s) - 16, 0) for s in streams])
    assert all(x == 0 for x in st), st
    return [o.tobytes()[:max(len(s) - 16, 0)] for o, s in zip(outs, streams)]


@pytest.mark.gpu
def test_ctr_extract_iv_classes_and_lengths(ctx, oracle):
    rnd = random.Random(11)
    key = os.urandom(32)
    lens = [0, 1, 15, 16, 17, 16 * 255, 16 * 256 + 3, 16 * (TILE_BLOCKS - 1), 16 * TILE_BLOCKS, 16 * (TILE_BLOCKS + 1),
            16 * 3 * TILE_BLOCKS + 7]
    plains, streams = [], []
    for low in IV_CLASSES:
        for n in lens:
            p = os.urandom(n)
            plains.append(p)
            streams.append(_stream(oracle, p, key, _iv(low, rnd)))
    assert _decode(ctx, streams, [key] * len(streams)) == plains


@pytest.mark.gpu
def test_ctr_extract_every_image_offset_and_run_phase(ctx, oracle):
    """Stream lengths 16 m + r for every r: the bodies start at every offset mod 16 of the uploaded image; IV low bytes
    across the whole range put run starts anywhere inside tiles."""
    rnd = random.Random(12)
    key = os.urandom(32)
    plains = [os.urandom(16 * rnd.randrange(1, 3 * TILE_BLOCKS) + r) for r in range(16) for _ in range(3)]
    streams = [_stream(oracle, p, key, _iv(bytes([rnd.randrange(256)]), rnd)) for p in plains]
    assert _decode(ctx, streams, [key] * len(streams)) == plains


@pytest.mark.gpu
def test_ctr_extract_split_bodies(ctx, oracle):
    """Streams over several bodies: boundaries inside the IV, inside a block, on block and tile boundaries."""
    rnd = random.Random(13)
    key = os.urandom(32)
    plains, streams, cuts = [], [], []
    for k in range(24):
        p = os.urandom(rnd.randrange(16, 4 * TILE_BLOCKS * 16))
        s = _stream(oracle, p, key, _iv(rnd.choice(IV_CLASSES), rnd))
        c = [rnd.randrange(1, 16), 16 + 16 * rnd.randrange(0, 50) + rnd.randrange(1, 16), 16 + 16 * TILE_BLOCKS,
             16 + 16 * TILE_BLOCKS + 5] + [rnd.randrange(1, len(s)) for _ in range(k % 6)]
        c += list(range(40, 40 + 3 * k, 3))   # runs of tiny bodies: several straddling blocks in a row
        plains.append(p); streams.append(s); cuts.append(c)
    assert _decode(ctx, streams, [key] * len(streams), cuts) == plains


@pytest.mark.gpu
def test_ctr_extract_interleaved_keys(ctx, oracle):
    rnd = random.Random(14)
    keys = [os.urandom(32) for _ in range(3)]
    plains = [os.urandom(rnd.randrange(0, 2 * TILE_BLOCKS * 16)) for _ in range(30)]
    ks = [keys[i % 3] for i in range(30)]
    streams = [_stream(oracle, p, k, _iv(rnd.choice(IV_CLASSES), rnd)) for p, k in zip(plains, ks)]
    assert _decode(ctx, streams, ks, [[rnd.randrange(1, max(len(s), 2))] for s in streams]) == plains


@pytest.mark.gpu
def test_ctr_create_matches_openssl(ctx, oracle):
    rnd = random.Random(15)
    ents = []
    for low in IV_CLASSES:
        for n in (0, 1, 17, 16 * 256 + 5, 16 * TILE_BLOCKS + 9):
            ents.append({"plain": os.urandom(n), "compression": 0, "encryption": 1, "cipher_mode": 1, "key": os.urandom(32),
                         "iv": _iv(low, rnd)})
    streams, _, st = ctx.encode_batch(ents)
    assert all(x == 0 for x in st), st
    for e, s in zip(ents, streams):
        assert s.tobytes() == e["iv"] + oracle.ctr(1, e["key"], e["iv"], e["plain"]), e["iv"].hex()
