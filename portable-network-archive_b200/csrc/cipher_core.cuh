// cipher_core.cuh -- AES-256 and Camellia-256 block primitives (table driven), host key schedules.
//
// Replaces, for the data-chunk path only, what the reference gets from the RustCrypto crates
// `aes 0.9.2` and `camellia 0.2.1` (not vendored under /root/reference; call sites
// lib/src/cipher.rs:21-55).  The algorithms are the published ones: FIPS-197 and RFC 3713.
// Pinned by tests against OpenSSL (oracle) and the reference KATs lib/src/cipher.rs:256-292.
//
// Word convention: the 16-byte block is four little-endian u32 words exactly as loaded from memory
// (AES column c = bytes 4c..4c+3, row r in bits 8r..8r+7).  Camellia works on big-endian 64-bit
// halves and byte-swaps at the edges.
#pragma once
#include "common.cuh"

namespace pna {

// ---------------------------------------------------------------------------------------------
// Table access policy.  On the device the 256-entry u32 tables are replicated 32x in shared memory
// (index*32 + lane) so that every lane owns a bank and lookups never conflict; on the host stride=1.
struct TabView {
    const uint32_t* t;
    uint32_t stride;  // 32 on device (replicated), 1 on host
    uint32_t lane;
    PNA_HD uint32_t operator()(uint32_t x) const { return t[x * stride + lane]; }
};

// ------------------------------------------------------------------------------------------ AES
struct AesTables {            // generated once on the host (aes_make_tables)
    uint32_t te0[256];        // (2s, s, s, 3s) rows 0..3, little-endian packed
    uint32_t td0[256];        // (0e.is, 09.is, 0d.is, 0b.is)
    uint8_t sbox[256];
    uint8_t inv_sbox[256];
};
struct AesKey {               // 15 round keys, encrypt order; dk = equivalent-inverse-cipher keys
    uint32_t rk[60];
    uint32_t dk[60];
};

inline uint8_t gf_mul(uint8_t a, uint8_t b) {
    uint8_t p = 0;
    for (int i = 0; i < 8; i++) {
        if (b & 1) p ^= a;
        uint8_t hi = a & 0x80;
        a = (uint8_t)(a << 1);
        if (hi) a ^= 0x1B;
        b >>= 1;
    }
    return p;
}
inline void aes_make_tables(AesTables* T) {
    // S-box: multiplicative inverse in GF(2^8) followed by the FIPS-197 affine map
    uint8_t inv[256];
    inv[0] = 0;
    for (int a = 1; a < 256; a++)
        for (int b = 1; b < 256; b++)
            if (gf_mul((uint8_t)a, (uint8_t)b) == 1) { inv[a] = (uint8_t)b; break; }
    for (int x = 0; x < 256; x++) {
        uint8_t v = inv[x], s = v;
        for (int k = 1; k <= 4; k++) s ^= (uint8_t)((v << k) | (v >> (8 - k)));
        s ^= 0x63;
        T->sbox[x] = s;
        T->inv_sbox[s] = (uint8_t)x;
    }
    for (int x = 0; x < 256; x++) {
        uint8_t s = T->sbox[x], is = T->inv_sbox[x];
        T->te0[x] = (uint32_t)gf_mul(s, 2) | ((uint32_t)s << 8) | ((uint32_t)s << 16) | ((uint32_t)gf_mul(s, 3) << 24);
        T->td0[x] = (uint32_t)gf_mul(is, 0x0e) | ((uint32_t)gf_mul(is, 0x09) << 8) |
                    ((uint32_t)gf_mul(is, 0x0d) << 16) | ((uint32_t)gf_mul(is, 0x0b) << 24);
    }
}
inline void aes256_expand_key(const AesTables* T, const uint8_t key[32], AesKey* K) {
    uint8_t w[240];
    memcpy(w, key, 32);
    uint8_t rcon = 1;
    for (int i = 8; i < 60; i++) {
        uint8_t t[4] = {w[4 * i - 4], w[4 * i - 3], w[4 * i - 2], w[4 * i - 1]};
        if (i % 8 == 0) {
            uint8_t r[4] = {T->sbox[t[1]], T->sbox[t[2]], T->sbox[t[3]], T->sbox[t[0]]};
            r[0] ^= rcon;
            rcon = gf_mul(rcon, 2);
            memcpy(t, r, 4);
        } else if (i % 8 == 4) {
            for (int k = 0; k < 4; k++) t[k] = T->sbox[t[k]];
        }
        for (int k = 0; k < 4; k++) w[4 * i + k] = w[4 * (i - 8) + k] ^ t[k];
    }
    for (int i = 0; i < 60; i++) K->rk[i] = load_le32(w + 4 * i);
    // equivalent inverse cipher: InvMixColumns on round keys 1..13
    for (int i = 0; i < 60; i++) {
        uint32_t v = K->rk[i];
        if (i >= 4 && i < 56) {
            uint32_t a = T->td0[T->sbox[v & 0xFF]], b = T->td0[T->sbox[(v >> 8) & 0xFF]],
                     c = T->td0[T->sbox[(v >> 16) & 0xFF]], d = T->td0[T->sbox[v >> 24]];
            v = a ^ rotl32(b, 8) ^ rotl32(c, 16) ^ rotl32(d, 24);
        }
        K->dk[i] = v;
    }
}

// The CTR / GCM keystream runs the cipher with the four rotations of Te0 as four tables (Te_K[x] = rotl(Te0[x], 8K)): no
// rotate per lookup.  A four-table view T4 provides  T4::at<K, B>(v) = Te_K[byte B of v].
// Host (and the CPU test tier): Te0 alone, rotated per lookup.
struct Te0Rot {
    const uint32_t* te0;
    template <int K, int B>
    PNA_HD uint32_t at(uint32_t v) const {
        const uint32_t e = te0[(v >> (8 * B)) & 0xFFu];
        return K ? rotl32(e, 8 * K) : e;
    }
};
#if defined(__CUDACC__) || defined(PNA_EMU)
// Device: the four tables replicated per lane in shared memory (128 KB), laid out [K >> 1][x][K & 1][lane].  The byte offset
// of a lookup is  x << 8 | lane * 4  (plus the table's constant): ONE byte permute builds it from the state word, and the
// table is picked by the load's immediate offset.  Lane l only ever reads bank l, so a warp's 32 lookups never conflict.
constexpr uint32_t AES_TE4_WORDS = 4 * 256 * 32;
__device__ __forceinline__ void aes_te4_fill(uint32_t* s_tab, const AesTables* aes) {
    for (uint32_t i = threadIdx.x; i < AES_TE4_WORDS; i += blockDim.x) {
        const uint32_t k = 2 * (i >> 14) + ((i >> 5) & 1);
        const uint32_t e = aes->te0[(i >> 6) & 255];
        s_tab[i] = k ? rotl32(e, 8 * k) : e;
    }
}
struct LaneTe4 {
    const uint8_t* tab;   // aes_te4_fill's tables
    uint32_t lane4;       // lane * 4
    template <int K, int B>
    __device__ __forceinline__ uint32_t at(uint32_t v) const {
        const uint32_t off = __byte_perm(v, lane4, 0x5504u | (B << 4));   // byte 0: lane4, byte 1: byte B of v, bytes 2-3: 0
        return *reinterpret_cast<const uint32_t*>(tab + ((K >> 1) * 65536 + (K & 1) * 128) + off);
    }
};
#endif

// Last-round bytes: the S-box byte of Te_K[x] sits at byte (1 + K) & 3.
PNA_HD uint32_t aes_last_bytes(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(__byte_perm(r0, r1, 0x0061u), __byte_perm(r2, r3, 0x4300u), 0x7610u);
#else
    return ((r0 >> 8) & 0xFFu) | ((r1 >> 8) & 0xFF00u) | ((r2 >> 8) & 0xFF0000u) | (r3 << 24);
#endif
}

// Rounds R0..13 and the last round on the columns a..d (which carry round key R0 - 1); rk = 60 words (any address space).
template <int R0, class T4>
PNA_HD void aes256_rounds4(uint32_t s[4], uint32_t a, uint32_t b, uint32_t c, uint32_t d, const uint32_t* rk, const T4& t) {
#pragma unroll
    for (int r = R0; r < 14; r++) {
        const uint32_t na = t.template at<0, 0>(a) ^ t.template at<1, 1>(b) ^ t.template at<2, 2>(c) ^ t.template at<3, 3>(d) ^ rk[4 * r + 0];
        const uint32_t nb = t.template at<0, 0>(b) ^ t.template at<1, 1>(c) ^ t.template at<2, 2>(d) ^ t.template at<3, 3>(a) ^ rk[4 * r + 1];
        const uint32_t nc = t.template at<0, 0>(c) ^ t.template at<1, 1>(d) ^ t.template at<2, 2>(a) ^ t.template at<3, 3>(b) ^ rk[4 * r + 2];
        const uint32_t nd = t.template at<0, 0>(d) ^ t.template at<1, 1>(a) ^ t.template at<2, 2>(b) ^ t.template at<3, 3>(c) ^ rk[4 * r + 3];
        a = na; b = nb; c = nc; d = nd;
    }
    s[0] = aes_last_bytes(t.template at<0, 0>(a), t.template at<1, 1>(b), t.template at<2, 2>(c), t.template at<3, 3>(d)) ^ rk[56];
    s[1] = aes_last_bytes(t.template at<0, 0>(b), t.template at<1, 1>(c), t.template at<2, 2>(d), t.template at<3, 3>(a)) ^ rk[57];
    s[2] = aes_last_bytes(t.template at<0, 0>(c), t.template at<1, 1>(d), t.template at<2, 2>(a), t.template at<3, 3>(b)) ^ rk[58];
    s[3] = aes_last_bytes(t.template at<0, 0>(d), t.template at<1, 1>(a), t.template at<2, 2>(b), t.template at<3, 3>(c)) ^ rk[59];
}
// s[4] in/out
template <class T4>
PNA_HD void aes256_encrypt_block4(uint32_t s[4], const uint32_t* rk, const T4& t) {
    aes256_rounds4<1>(s, s[0] ^ rk[0], s[1] ^ rk[1], s[2] ^ rk[2], s[3] ^ rk[3], rk, t);
}

// AES-256-CTR over a counter run: up to 256 consecutive counter blocks that share bytes 0..14 (only the low byte x, byte 15,
// counts).  Byte 15 is byte 3 of column d, so in round 1 it reaches one lookup (column a's Te3) and in round 2 it reaches,
// through round-1 column a, one lookup per column.  aes256_ctr_run_init computes once per run everything else of rounds 1-2
// (27 lookups): p[0] = round-1 column a without its Te3 term, p[1..4] = round-2 columns a..d without their term in round-1
// column a.  aes256_ctr_run_block then encrypts the run's block x with 5 lookups for rounds 1-2 instead of 32.
template <class T4>
PNA_HD void aes256_ctr_run_init(const uint32_t ctr[4], const uint32_t* rk, const T4& t, uint32_t p[5]) {
    const uint32_t a = ctr[0] ^ rk[0], b = ctr[1] ^ rk[1], c = ctr[2] ^ rk[2], d = ctr[3] ^ rk[3];
    p[0] = t.template at<0, 0>(a) ^ t.template at<1, 1>(b) ^ t.template at<2, 2>(c) ^ rk[4];
    const uint32_t b1 = t.template at<0, 0>(b) ^ t.template at<1, 1>(c) ^ t.template at<2, 2>(d) ^ t.template at<3, 3>(a) ^ rk[5];
    const uint32_t c1 = t.template at<0, 0>(c) ^ t.template at<1, 1>(d) ^ t.template at<2, 2>(a) ^ t.template at<3, 3>(b) ^ rk[6];
    const uint32_t d1 = t.template at<0, 0>(d) ^ t.template at<1, 1>(a) ^ t.template at<2, 2>(b) ^ t.template at<3, 3>(c) ^ rk[7];
    p[1] = t.template at<1, 1>(b1) ^ t.template at<2, 2>(c1) ^ t.template at<3, 3>(d1) ^ rk[8];    // lacks Te0[a1 byte 0]
    p[2] = t.template at<0, 0>(b1) ^ t.template at<1, 1>(c1) ^ t.template at<2, 2>(d1) ^ rk[9];    // lacks Te3[a1 byte 3]
    p[3] = t.template at<0, 0>(c1) ^ t.template at<1, 1>(d1) ^ t.template at<3, 3>(b1) ^ rk[10];   // lacks Te2[a1 byte 2]
    p[4] = t.template at<0, 0>(d1) ^ t.template at<2, 2>(b1) ^ t.template at<3, 3>(c1) ^ rk[11];   // lacks Te1[a1 byte 1]
}
// x24 = the block's counter low byte in bits 24..31 (other bits zero); s = E_K(counter)
template <class T4>
PNA_HD void aes256_ctr_run_block(const uint32_t p[5], uint32_t x24, const uint32_t* rk, const T4& t, uint32_t s[4]) {
    const uint32_t a1 = p[0] ^ t.template at<3, 3>(x24 ^ rk[3]);
    aes256_rounds4<3>(s, p[1] ^ t.template at<0, 0>(a1), p[2] ^ t.template at<3, 3>(a1), p[3] ^ t.template at<2, 2>(a1),
                      p[4] ^ t.template at<1, 1>(a1), rk, t);
}

template <class Tab>
PNA_HD void aes256_encrypt_block(uint32_t s[4], const uint32_t* rk, const Tab& te) {
    uint32_t a = s[0] ^ rk[0], b = s[1] ^ rk[1], c = s[2] ^ rk[2], d = s[3] ^ rk[3];
#pragma unroll
    for (int r = 1; r < 14; r++) {
        uint32_t na = te(a & 0xFF) ^ rotl32(te((b >> 8) & 0xFF), 8) ^ rotl32(te((c >> 16) & 0xFF), 16) ^
                      rotl32(te(d >> 24), 24) ^ rk[4 * r + 0];
        uint32_t nb = te(b & 0xFF) ^ rotl32(te((c >> 8) & 0xFF), 8) ^ rotl32(te((d >> 16) & 0xFF), 16) ^
                      rotl32(te(a >> 24), 24) ^ rk[4 * r + 1];
        uint32_t nc = te(c & 0xFF) ^ rotl32(te((d >> 8) & 0xFF), 8) ^ rotl32(te((a >> 16) & 0xFF), 16) ^
                      rotl32(te(b >> 24), 24) ^ rk[4 * r + 2];
        uint32_t nd = te(d & 0xFF) ^ rotl32(te((a >> 8) & 0xFF), 8) ^ rotl32(te((b >> 16) & 0xFF), 16) ^
                      rotl32(te(c >> 24), 24) ^ rk[4 * r + 3];
        a = na; b = nb; c = nc; d = nd;
    }
#define PNA_SB(x) ((te(x) >> 8) & 0xFFu)
    s[0] = (PNA_SB(a & 0xFF) | (PNA_SB((b >> 8) & 0xFF) << 8) | (PNA_SB((c >> 16) & 0xFF) << 16) | (PNA_SB(d >> 24) << 24)) ^ rk[56];
    s[1] = (PNA_SB(b & 0xFF) | (PNA_SB((c >> 8) & 0xFF) << 8) | (PNA_SB((d >> 16) & 0xFF) << 16) | (PNA_SB(a >> 24) << 24)) ^ rk[57];
    s[2] = (PNA_SB(c & 0xFF) | (PNA_SB((d >> 8) & 0xFF) << 8) | (PNA_SB((a >> 16) & 0xFF) << 16) | (PNA_SB(b >> 24) << 24)) ^ rk[58];
    s[3] = (PNA_SB(d & 0xFF) | (PNA_SB((a >> 8) & 0xFF) << 8) | (PNA_SB((b >> 16) & 0xFF) << 16) | (PNA_SB(c >> 24) << 24)) ^ rk[59];
#undef PNA_SB
}
// dk = equivalent-inverse keys (AesKey::dk); isb = inverse S-box bytes (256)
template <class Tab>
PNA_HD void aes256_decrypt_block(uint32_t s[4], const uint32_t* dk, const Tab& td, const uint8_t* isb) {
    uint32_t a = s[0] ^ dk[56], b = s[1] ^ dk[57], c = s[2] ^ dk[58], d = s[3] ^ dk[59];
#pragma unroll
    for (int r = 13; r >= 1; r--) {
        uint32_t na = td(a & 0xFF) ^ rotl32(td((d >> 8) & 0xFF), 8) ^ rotl32(td((c >> 16) & 0xFF), 16) ^
                      rotl32(td(b >> 24), 24) ^ dk[4 * r + 0];
        uint32_t nb = td(b & 0xFF) ^ rotl32(td((a >> 8) & 0xFF), 8) ^ rotl32(td((d >> 16) & 0xFF), 16) ^
                      rotl32(td(c >> 24), 24) ^ dk[4 * r + 1];
        uint32_t nc = td(c & 0xFF) ^ rotl32(td((b >> 8) & 0xFF), 8) ^ rotl32(td((a >> 16) & 0xFF), 16) ^
                      rotl32(td(d >> 24), 24) ^ dk[4 * r + 2];
        uint32_t nd = td(d & 0xFF) ^ rotl32(td((c >> 8) & 0xFF), 8) ^ rotl32(td((b >> 16) & 0xFF), 16) ^
                      rotl32(td(a >> 24), 24) ^ dk[4 * r + 3];
        a = na; b = nb; c = nc; d = nd;
    }
    s[0] = ((uint32_t)isb[a & 0xFF] | ((uint32_t)isb[(d >> 8) & 0xFF] << 8) | ((uint32_t)isb[(c >> 16) & 0xFF] << 16) | ((uint32_t)isb[b >> 24] << 24)) ^ dk[0];
    s[1] = ((uint32_t)isb[b & 0xFF] | ((uint32_t)isb[(a >> 8) & 0xFF] << 8) | ((uint32_t)isb[(d >> 16) & 0xFF] << 16) | ((uint32_t)isb[c >> 24] << 24)) ^ dk[1];
    s[2] = ((uint32_t)isb[c & 0xFF] | ((uint32_t)isb[(b >> 8) & 0xFF] << 8) | ((uint32_t)isb[(a >> 16) & 0xFF] << 16) | ((uint32_t)isb[d >> 24] << 24)) ^ dk[2];
    s[3] = ((uint32_t)isb[d & 0xFF] | ((uint32_t)isb[(c >> 8) & 0xFF] << 8) | ((uint32_t)isb[(b >> 16) & 0xFF] << 16) | ((uint32_t)isb[a >> 24] << 24)) ^ dk[3];
}

// ------------------------------------------------------------------------------------- Camellia
// RFC 3713.  F(x,k) = P(S(x^k)); the eight byte lanes are pre-combined into 8 SP tables of 64-bit
// entries, stored as (hi,lo) u32 pairs: sp[i][b] = P applied to S_i[b] placed in byte lane i.
struct CamelliaTables {
    uint32_t sp_hi[8][256];
    uint32_t sp_lo[8][256];
};
struct CamelliaKey {
    // subkeys in encryption order: kw1,kw2, k1..k6, ke1,ke2, k7..k12, ke3,ke4, k13..k18, ke5,ke6, k19..k24, kw3,kw4
    uint64_t ek[34];
    uint64_t dk[34];  // same sequence for decryption
};

static const uint8_t CAMELLIA_SBOX1[256] = {
    112, 130, 44,  236, 179, 39,  192, 229, 228, 133, 87,  53,  234, 12,  174, 65,  35,  239, 107, 147, 69,  25,
    165, 33,  237, 14,  79,  78,  29,  101, 146, 189, 134, 184, 175, 143, 124, 235, 31,  206, 62,  48,  220, 95,
    94,  197, 11,  26,  166, 225, 57,  202, 213, 71,  93,  61,  217, 1,   90,  214, 81,  86,  108, 77,  139, 13,
    154, 102, 251, 204, 176, 45,  116, 18,  43,  32,  240, 177, 132, 153, 223, 76,  203, 194, 52,  126, 118, 5,
    109, 183, 169, 49,  209, 23,  4,   215, 20,  88,  58,  97,  222, 27,  17,  28,  50,  15,  156, 22,  83,  24,
    242, 34,  254, 68,  207, 178, 195, 181, 122, 145, 36,  8,   232, 168, 96,  252, 105, 80,  170, 208, 160, 125,
    161, 137, 98,  151, 84,  91,  30,  149, 224, 255, 100, 210, 16,  196, 0,   72,  163, 247, 117, 219, 138, 3,
    230, 218, 9,   63,  221, 148, 135, 92,  131, 2,   205, 74,  144, 51,  115, 103, 246, 243, 157, 127, 191, 226,
    82,  155, 216, 38,  200, 55,  198, 59,  129, 150, 111, 75,  19,  190, 99,  46,  233, 121, 167, 140, 159, 110,
    188, 142, 41,  245, 249, 182, 47,  253, 180, 89,  120, 152, 6,   106, 231, 70,  113, 186, 212, 37,  171, 66,
    136, 162, 141, 250, 114, 7,   185, 85,  248, 238, 172, 10,  54,  73,  42,  104, 60,  56,  241, 164, 64,  40,
    211, 123, 187, 201, 67,  193, 21,  227, 173, 244, 119, 199, 128, 158};

inline void camellia_make_tables(CamelliaTables* T) {
    // which outputs y1..y8 each input lane t1..t8 feeds (RFC 3713 section 2.4.1, P-function)
    static const uint8_t feeds[8] = {
        /* t1 -> y1 y2 y3 y5 y8 */ 0x80 | 0x40 | 0x20 | 0x08 | 0x01,
        /* t2 -> y2 y3 y4 y5 y6 */ 0x40 | 0x20 | 0x10 | 0x08 | 0x04,
        /* t3 -> y1 y3 y4 y6 y7 */ 0x80 | 0x20 | 0x10 | 0x04 | 0x02,
        /* t4 -> y1 y2 y4 y7 y8 */ 0x80 | 0x40 | 0x10 | 0x02 | 0x01,
        /* t5 -> y2 y3 y4 y6 y7 y8 */ 0x40 | 0x20 | 0x10 | 0x04 | 0x02 | 0x01,
        /* t6 -> y1 y3 y4 y5 y7 y8 */ 0x80 | 0x20 | 0x10 | 0x08 | 0x02 | 0x01,
        /* t7 -> y1 y2 y4 y5 y6 y8 */ 0x80 | 0x40 | 0x10 | 0x08 | 0x04 | 0x01,
        /* t8 -> y1 y2 y3 y5 y6 y7 */ 0x80 | 0x40 | 0x20 | 0x08 | 0x04 | 0x02,
    };
    for (int lane = 0; lane < 8; lane++)
        for (int x = 0; x < 256; x++) {
            uint8_t s1 = CAMELLIA_SBOX1[x];
            uint8_t s;
            switch (lane) {  // t1:S1 t2:S2 t3:S3 t4:S4 t5:S2 t6:S3 t7:S4 t8:S1
                case 0: case 7: s = s1; break;
                case 1: case 4: s = (uint8_t)((s1 << 1) | (s1 >> 7)); break;
                case 2: case 5: s = (uint8_t)((s1 << 7) | (s1 >> 1)); break;
                default: s = CAMELLIA_SBOX1[(uint8_t)((x << 1) | (x >> 7))]; break;
            }
            uint64_t v = 0;
            for (int y = 0; y < 8; y++)
                if (feeds[lane] & (0x80 >> y)) v |= (uint64_t)s << (56 - 8 * y);
            T->sp_hi[lane][x] = (uint32_t)(v >> 32);
            T->sp_lo[lane][x] = (uint32_t)v;
        }
}

// F on a 64-bit half given as (hi,lo).  hi_t/lo_t index [lane*256 + byte].
PNA_HD void camellia_f(uint32_t xh, uint32_t xl, uint32_t kh, uint32_t kl, const uint32_t* hi_t, const uint32_t* lo_t,
                       uint32_t& oh, uint32_t& ol) {
    xh ^= kh; xl ^= kl;
    uint32_t i0 = xh >> 24, i1 = 256 + ((xh >> 16) & 0xFF), i2 = 512 + ((xh >> 8) & 0xFF), i3 = 768 + (xh & 0xFF);
    uint32_t i4 = 1024 + (xl >> 24), i5 = 1280 + ((xl >> 16) & 0xFF), i6 = 1536 + ((xl >> 8) & 0xFF), i7 = 1792 + (xl & 0xFF);
    oh = hi_t[i0] ^ hi_t[i1] ^ hi_t[i2] ^ hi_t[i3] ^ hi_t[i4] ^ hi_t[i5] ^ hi_t[i6] ^ hi_t[i7];
    ol = lo_t[i0] ^ lo_t[i1] ^ lo_t[i2] ^ lo_t[i3] ^ lo_t[i4] ^ lo_t[i5] ^ lo_t[i6] ^ lo_t[i7];
}
inline uint64_t camellia_f64(const CamelliaTables* T, uint64_t x, uint64_t k) {
    uint32_t oh, ol;
    camellia_f((uint32_t)(x >> 32), (uint32_t)x, (uint32_t)(k >> 32), (uint32_t)k, &T->sp_hi[0][0], &T->sp_lo[0][0], oh, ol);
    return ((uint64_t)oh << 32) | ol;
}
inline void rot128(uint64_t hi, uint64_t lo, int n, uint64_t& oh, uint64_t& ol) {  // rotate left by n (0..127)
    n &= 127;
    if (n >= 64) { uint64_t t = hi; hi = lo; lo = t; n -= 64; }
    if (n == 0) { oh = hi; ol = lo; return; }
    oh = (hi << n) | (lo >> (64 - n));
    ol = (lo << n) | (hi >> (64 - n));
}
inline uint64_t load_be64(const uint8_t* p) {
    uint64_t v = 0;
    for (int i = 0; i < 8; i++) v = (v << 8) | p[i];
    return v;
}
inline void camellia256_expand_key(const CamelliaTables* T, const uint8_t key[32], CamelliaKey* K) {
    const uint64_t S1 = 0xA09E667F3BCC908BULL, S2 = 0xB67AE8584CAA73B2ULL, S3 = 0xC6EF372FE94F82BEULL,
                   S4 = 0x54FF53A5F1D36F1CULL, S5 = 0x10E527FADE682D1DULL, S6 = 0xB05688C2B3E6C1FDULL;
    uint64_t KLh = load_be64(key), KLl = load_be64(key + 8), KRh = load_be64(key + 16), KRl = load_be64(key + 24);
    uint64_t D1 = KLh ^ KRh, D2 = KLl ^ KRl;
    D2 ^= camellia_f64(T, D1, S1);
    D1 ^= camellia_f64(T, D2, S2);
    D1 ^= KLh; D2 ^= KLl;
    D2 ^= camellia_f64(T, D1, S3);
    D1 ^= camellia_f64(T, D2, S4);
    uint64_t KAh = D1, KAl = D2;
    D1 = KAh ^ KRh; D2 = KAl ^ KRl;
    D2 ^= camellia_f64(T, D1, S5);
    D1 ^= camellia_f64(T, D2, S6);
    uint64_t KBh = D1, KBl = D2;
    uint64_t* e = K->ek;
    auto put = [&](int idx, uint64_t h, uint64_t l, int n) { rot128(h, l, n, e[idx], e[idx + 1]); };
    put(0, KLh, KLl, 0);     // kw1 kw2
    put(2, KBh, KBl, 0);     // k1 k2
    put(4, KRh, KRl, 15);    // k3 k4
    put(6, KAh, KAl, 15);    // k5 k6
    put(8, KRh, KRl, 30);    // ke1 ke2
    put(10, KBh, KBl, 30);   // k7 k8
    put(12, KLh, KLl, 45);   // k9 k10
    put(14, KAh, KAl, 45);   // k11 k12
    put(16, KLh, KLl, 60);   // ke3 ke4
    put(18, KRh, KRl, 60);   // k13 k14
    put(20, KBh, KBl, 60);   // k15 k16
    put(22, KLh, KLl, 77);   // k17 k18
    put(24, KAh, KAl, 77);   // ke5 ke6
    put(26, KRh, KRl, 94);   // k19 k20
    put(28, KAh, KAl, 94);   // k21 k22
    put(30, KLh, KLl, 111);  // k23 k24
    put(32, KBh, KBl, 111);  // kw3 kw4
    // decryption = same network with the subkey order reversed (RFC 3713 2.3.2)
    uint64_t* d = K->dk;
    d[0] = e[32]; d[1] = e[33];
    d[32] = e[0]; d[33] = e[1];
    // body positions 2..31: rounds and FL pairs mirrored
    for (int i = 0; i < 30; i++) d[2 + i] = e[31 - i];
}

// one block; subkeys k[34] as u64 (any address space); block words LE as loaded; tables in hi_t/lo_t
PNA_HD void camellia256_crypt_block(uint32_t s[4], const uint64_t* k, const uint32_t* hi_t, const uint32_t* lo_t) {
    uint32_t d1h = bswap32(s[0]), d1l = bswap32(s[1]), d2h = bswap32(s[2]), d2l = bswap32(s[3]);
    d1h ^= (uint32_t)(k[0] >> 32); d1l ^= (uint32_t)k[0];
    d2h ^= (uint32_t)(k[1] >> 32); d2l ^= (uint32_t)k[1];
    int ki = 2;
#pragma unroll 1
    for (int grp = 0; grp < 4; grp++) {
#pragma unroll
        for (int r = 0; r < 3; r++) {
            uint32_t oh, ol;
            uint64_t ka = k[ki], kb = k[ki + 1];
            camellia_f(d1h, d1l, (uint32_t)(ka >> 32), (uint32_t)ka, hi_t, lo_t, oh, ol);
            d2h ^= oh; d2l ^= ol;
            camellia_f(d2h, d2l, (uint32_t)(kb >> 32), (uint32_t)kb, hi_t, lo_t, oh, ol);
            d1h ^= oh; d1l ^= ol;
            ki += 2;
        }
        if (grp < 3) {
            uint64_t ke_a = k[ki], ke_b = k[ki + 1];
            ki += 2;
            // FL on D1
            d1l ^= rotl32(d1h & (uint32_t)(ke_a >> 32), 1);
            d1h ^= (d1l | (uint32_t)ke_a);
            // FLINV on D2
            d2h ^= (d2l | (uint32_t)ke_b);
            d2l ^= rotl32(d2h & (uint32_t)(ke_b >> 32), 1);
        }
    }
    d2h ^= (uint32_t)(k[32] >> 32); d2l ^= (uint32_t)k[32];
    d1h ^= (uint32_t)(k[33] >> 32); d1l ^= (uint32_t)k[33];
    s[0] = bswap32(d2h); s[1] = bswap32(d2l); s[2] = bswap32(d1h); s[3] = bswap32(d1l);
}

// 128-bit big-endian counter add on LE-loaded words (ctr 0.10.1 Ctr128BE: IV + block index)
PNA_HD void ctr128be_add(const uint32_t iv[4], uint64_t add, uint32_t out[4]) {
    uint32_t w3 = bswap32(iv[3]), w2 = bswap32(iv[2]), w1 = bswap32(iv[1]), w0 = bswap32(iv[0]);
    uint64_t lo = ((uint64_t)w2 << 32) | w3, hi = ((uint64_t)w0 << 32) | w1;
    uint64_t nlo = lo + add;
    if (nlo < lo) hi += 1;
    out[3] = bswap32((uint32_t)nlo); out[2] = bswap32((uint32_t)(nlo >> 32));
    out[1] = bswap32((uint32_t)hi); out[0] = bswap32((uint32_t)(hi >> 32));
}

}  // namespace pna
