// zstd_core.cuh -- Zstandard (RFC 8878) frame/block parsing, FSE + Huffman table construction and
// the serial entropy decoders, written as PNA_HD code shared by the sm_100a kernels
// (zstd_kernels.cuh) and the g++ host test build (tests/host/host_core.cpp).
//
// Replaces `zstd::Decoder::with_buffer` at /root/reference/lib/src/entry/read.rs:181
// (crate zstd 0.13.3 -> zstd-sys 2.0.14+zstd.1.5.7, C libzstd; not vendored under /root/reference).
// The format is the published one; behaviour on malformed input follows libzstd's checks where noted.
//
// Decode plan (see DESIGN.md): scan frames -> parse blocks -> resolve repeat/treeless table sources
// -> per block entropy decode (literals + sequences, block-parallel) -> per frame prefix (output
// offsets, repeat-offset history) -> LZ execution.
#pragma once
#include "common.cuh"

namespace pna {
namespace zs {

constexpr uint32_t MAGIC = 0xFD2FB528u;
constexpr uint32_t BLOCK_MAX = 128 * 1024;
constexpr int HUF_LOG_MAX = 12;
constexpr int LL_LOG_MAX = 9, OF_LOG_MAX = 8, ML_LOG_MAX = 9;
constexpr int LL_MAXSYM = 35, OF_MAXSYM = 31, ML_MAXSYM = 52;
constexpr uint32_t WINDOW_MAX = 1u << 27;  // ZSTD_WINDOWLOG_LIMIT_DEFAULT used by the streaming decoder
constexpr uint32_t REP_SYM = 0x80000000u;  // symbolic repeat-offset marker (slot in bits 30-29, delta below)

enum : uint8_t { BT_RAW = 0, BT_RLE = 1, BT_COMPRESSED = 2 };
enum : uint8_t { LT_RAW = 0, LT_RLE = 1, LT_COMPRESSED = 2, LT_TREELESS = 3 };
enum : uint8_t { SM_PREDEF = 0, SM_RLE = 1, SM_FSE = 2, SM_REPEAT = 3 };

struct ZBlock {
    uint64_t src;       // byte offset of the block content inside the comp arena
    uint64_t out_off;   // absolute offset in the out arena (prefix pass)
    uint64_t frame_out; // absolute offset in the out arena where this block's frame starts
    uint64_t lit_off;   // literal arena offset (Huffman literals only)
    uint64_t seq_off;   // first sequence slot in the sequence arrays
    uint32_t entry;
    uint32_t size;      // block content size; RLE: regenerated size
    uint32_t out_size;  // regenerated size (raw/RLE from header, compressed from the entropy pass)
    uint32_t lit_regen, lit_csize, lit_pos;   // lit_pos: offset of the literal payload inside the block
    uint32_t nseq;
    uint32_t seq_pos;   // offset (inside block) of the first table description / bitstream after the modes byte
    uint32_t desc[3];   // offset (inside block) of the LL/OF/ML description (FSE NCount or RLE symbol)
    uint32_t bs_pos, bs_len;  // sequence bitstream
    int32_t tsrc[3];    // block index whose description builds the LL/OF/ML table (repeat resolved); -1 = predefined
    int32_t huf_src;    // block index whose Huffman tree description applies
    uint32_t rep_out[3];  // outgoing repeat-offset history, possibly symbolic in the incoming one
    uint32_t rep_in[3];   // incoming history, absolute (prefix pass)
    uint32_t lit_used;    // sum of literal lengths consumed by sequences
    uint8_t type, first_in_frame, lit_type, lit_streams;
    uint8_t mode[3];
    uint8_t _pad;
    int32_t status;
    uint32_t esc_n;                    // sequences whose ll or ml did not fit 16 bits (SeqRec escapes)
    uint32_t esc_idx[4], esc_ll[4], esc_ml[4];
};

// ---------------------------------------------------------------------------------------------
// Little-endian bit array view over an arena (aligned u32 words, padded by >= 8 bytes at the end).
PNA_HD uint32_t peek_bits(const uint32_t* w, uint64_t bitpos, int n) {  // 0 <= n <= 32
    uint64_t wi = bitpos >> 5;
    uint32_t sh = (uint32_t)bitpos & 31u;
    uint64_t v = (((uint64_t)w[wi + 1] << 32) | w[wi]) >> sh;
    return n >= 32 ? (uint32_t)v : ((uint32_t)v & ((1u << n) - 1u));
}

// Backward bitstream over bytes [begin, begin+len) of the arena.  pos counts the unread bits.
struct BackBits {
    const uint32_t* w;
    uint64_t base;   // bit address of `begin`
    int64_t pos;     // remaining bits; < 0 after an over-read
    PNA_HD bool init(const uint32_t* words, const uint8_t* bytes, uint64_t begin, uint64_t len) {
        w = words;
        base = begin * 8;
        pos = 0;
        if (len == 0) return false;
        uint8_t last = bytes[begin + len - 1];
        if (last == 0) return false;
        pos = (int64_t)(len - 1) * 8 + highbit32(last);
        return true;
    }
    PNA_HD uint32_t read(int n) {  // missing bits below the start read as zero
        pos -= n;
        if (pos >= 0) return peek_bits(w, base + (uint64_t)pos, n);
        int have = n + (int)pos;  // bits that actually exist
        if (have <= 0) return 0;
        return peek_bits(w, base, have) << (n - have);
    }
    PNA_HD uint32_t peek_top(int n) const {  // look at the next n bits without consuming (zero filled)
        if (pos >= n) return peek_bits(w, base + (uint64_t)(pos - n), n);
        if (pos <= 0) return 0;
        return peek_bits(w, base, (int)pos) << (n - (int)pos);
    }
};

// Forward (LSB first) bit reader over bytes, bounds checked, used for FSE table descriptions.
struct FwdBits {
    const uint8_t* p;
    uint32_t avail;   // bytes available
    uint32_t bit;     // bits consumed
    PNA_HD uint32_t peek32() const {
        uint32_t byte = bit >> 3, sh = bit & 7;
        uint64_t v = 0;
#pragma unroll
        for (int i = 0; i < 5; i++)
            if (byte + i < avail) v |= (uint64_t)p[byte + i] << (8 * i);
        return (uint32_t)(v >> sh);
    }
};

// ---------------------------------------------------------------------------------------------
// FSE table description (libzstd FSE_readNCount semantics).  Returns bytes consumed or -1.
PNA_HD int fse_read_ncount(const uint8_t* p, uint32_t avail, int max_sym, int max_log, int16_t* norm, int* table_log,
                           int* n_sym) {
    if (avail < 1) return -1;
    FwdBits fb{p, avail, 0};
    uint32_t bs = fb.peek32();
    int nb = (int)(bs & 0xF) + 5;
    if (nb > max_log) return -1;
    *table_log = nb;
    fb.bit += 4;
    int remaining = (1 << nb) + 1;
    int threshold = 1 << nb;
    nb++;
    int sym = 0;
    bool prev0 = false;
    const int max_sv1 = max_sym + 1;
    for (;;) {
        if (prev0) {
            for (;;) {
                uint32_t two = fb.peek32() & 3u;
                fb.bit += 2;
                int to = sym + (int)two;   // symbols skipped carry probability 0
                for (; sym < to && sym < max_sv1; sym++) norm[sym] = 0;
                sym = to;                  // may run past the alphabet: rejected below
                if (two != 3) break;
                if (fb.bit > avail * 8 + 32) return -1;
            }
            if (sym >= max_sv1) break;
        }
        {
            bs = fb.peek32();
            int mx = (2 * threshold - 1) - remaining;
            int count;
            if ((int)(bs & (uint32_t)(threshold - 1)) < mx) {
                count = (int)(bs & (uint32_t)(threshold - 1));
                fb.bit += nb - 1;
            } else {
                count = (int)(bs & (uint32_t)(2 * threshold - 1));
                if (count >= threshold) count -= mx;
                fb.bit += nb;
            }
            count--;
            if (count >= 0) remaining -= count; else remaining += count;
            norm[sym++] = (int16_t)count;
            prev0 = (count == 0);
            if (remaining < threshold) {
                if (remaining <= 1) break;
                nb = highbit32((uint32_t)remaining) + 1;
                threshold = 1 << (nb - 1);
            }
            if (sym >= max_sv1) break;
        }
    }
    if (remaining != 1) return -1;
    if (sym > max_sv1) return -1;
    int bytes = (int)((fb.bit + 7) >> 3);
    if ((uint32_t)bytes > avail) return -1;
    *n_sym = sym;
    return bytes;
}

// Sequence FSE decode entry: 8 bytes, base value and extra-bit count folded in (one lookup per code).
struct SeqEntry {
    uint16_t next;     // new-state base
    uint8_t nb_extra;  // additional bits of the code's value
    uint8_t nb;        // state bits to read
    uint32_t base;     // value baseline
};
struct FseEntry {  // plain FSE (Huffman weights): 4 bytes
    uint16_t next;
    uint8_t sym;
    uint8_t nb;
};

PNA_HD uint32_t ll_base(int c) {
    return c < 16 ? (uint32_t)c
         : c < 20 ? (uint32_t)(16 + 2 * (c - 16))
         : c < 22 ? (uint32_t)(24 + 4 * (c - 20))
         : c < 24 ? (uint32_t)(32 + 8 * (c - 22))
         : c == 24 ? 48u : (1u << (c - 19));   // 25->64, 26->128 ... 35->65536
}
PNA_HD int ll_bits(int c) {
    return c < 16 ? 0 : c < 20 ? 1 : c < 22 ? 2 : c < 24 ? 3 : c == 24 ? 4 : c == 25 ? 6 : (c - 19);
}
PNA_HD uint32_t ml_base(int c) {
    return c < 32 ? (uint32_t)(c + 3)
         : c < 36 ? (uint32_t)(35 + 2 * (c - 32))
         : c < 38 ? (uint32_t)(43 + 4 * (c - 36))
         : c < 40 ? (uint32_t)(51 + 8 * (c - 38))
         : c < 42 ? (uint32_t)(67 + 16 * (c - 40))
         : c == 42 ? 99u : ((1u << (c - 36)) + 3u);  // 43->131, 44->259 ... 52->65539
}
PNA_HD int ml_bits(int c) {
    return c < 32 ? 0 : c < 36 ? 1 : c < 38 ? 2 : c < 40 ? 3 : c < 42 ? 4 : c == 42 ? 5 : (c - 36);
}

// predefined distributions (RFC 8878 3.1.1.3.2.2)
PNA_HD int predef_norm(int kind, int s) {
    if (kind == 0) {  // LL, log 6
        return s == 0 ? 4 : s == 1 ? 3 : s < 13 ? 2 : s < 16 ? 1 : s < 25 ? 2 : s == 25 ? 3 : s == 26 ? 2
             : s < 32 ? 1 : -1;
    }
    if (kind == 1) {  // OF, log 5
        return s < 6 ? 1 : s < 9 ? 2 : s < 24 ? 1 : -1;
    }
    // ML, log 6
    return s == 0 ? 1 : s == 1 ? 4 : s == 2 ? 3 : s < 9 ? 2 : s < 46 ? 1 : -1;
}

// Build a sequence decoding table from normalized counts.  kind: 0 LL, 1 OF, 2 ML.
// scratch: uint16_t[53] symbolNext.  tab must hold 1<<log entries.
PNA_HD void fse_build_seq_table(SeqEntry* tab, const int16_t* norm, int n_sym, int log, int kind, uint16_t* next_of) {
    const int size = 1 << log;
    int high = size - 1;
    for (int s = 0; s < n_sym; s++) {
        if (norm[s] == -1) { tab[high--].base = (uint32_t)s; next_of[s] = 1; }
        else next_of[s] = (uint16_t)norm[s];
    }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < n_sym; s++) {
        for (int i = 0; i < norm[s]; i++) {
            tab[pos].base = (uint32_t)s;
            pos = (pos + step) & mask;
            while (pos > high) pos = (pos + step) & mask;
        }
    }
    for (int u = 0; u < size; u++) {
        int s = (int)tab[u].base;
        uint32_t ns = next_of[s]++;
        int nb = log - highbit32(ns);
        SeqEntry e;
        e.nb = (uint8_t)nb;
        e.next = (uint16_t)((ns << nb) - (uint32_t)size);
        if (kind == 0) { e.base = ll_base(s); e.nb_extra = (uint8_t)ll_bits(s); }
        else if (kind == 1) { e.base = 1u << s; e.nb_extra = (uint8_t)s; }   // offset_value = (1<<code) + bits
        else { e.base = ml_base(s); e.nb_extra = (uint8_t)ml_bits(s); }
        tab[u] = e;
    }
}
PNA_HD void fse_rle_seq_table(SeqEntry* tab, int s, int kind) {
    SeqEntry e;
    e.nb = 0; e.next = 0;
    if (kind == 0) { e.base = ll_base(s); e.nb_extra = (uint8_t)ll_bits(s); }
    else if (kind == 1) { e.base = 1u << s; e.nb_extra = (uint8_t)s; }
    else { e.base = ml_base(s); e.nb_extra = (uint8_t)ml_bits(s); }
    tab[0] = e;
}

// Build the table for one symbol kind of block `b` from its (already resolved) source block.
// Returns the accuracy log, or -1 on corruption.
PNA_HD int seq_table_for(const uint8_t* comp, const ZBlock* blocks, const ZBlock& b, int kind, SeqEntry* tab,
                         int16_t* norm, uint16_t* next_of) {
    const int max_sym = kind == 0 ? LL_MAXSYM : kind == 1 ? OF_MAXSYM : ML_MAXSYM;
    const int max_log = kind == 0 ? LL_LOG_MAX : kind == 1 ? OF_LOG_MAX : ML_LOG_MAX;
    int src = b.tsrc[kind];
    if (src < 0) {  // predefined
        int log = kind == 1 ? 5 : 6;
        int n = kind == 0 ? 36 : kind == 1 ? 29 : 53;
        for (int s = 0; s < n; s++) norm[s] = (int16_t)predef_norm(kind, s);
        fse_build_seq_table(tab, norm, n, log, kind, next_of);
        return log;
    }
    const ZBlock& sb = blocks[src];
    const uint8_t* d = comp + sb.src + sb.desc[kind];
    uint32_t avail = sb.size - sb.desc[kind];
    if (sb.mode[kind] == SM_RLE) {
        if (avail < 1 || d[0] > max_sym) return -1;
        fse_rle_seq_table(tab, d[0], kind);
        return 0;
    }
    int log = 0, n_sym = 0;
    if (fse_read_ncount(d, avail, max_sym, max_log, norm, &log, &n_sym) < 0) return -1;
    fse_build_seq_table(tab, norm, n_sym, log, kind, next_of);
    return log;
}

// ---------------------------------------------------------------------------------------------
// Compact sequence tables for the lane-per-block decoder (kernels_zstd.cuh zstd_seq_kernel): one
// 16-bit entry per state = code << 10 | ns, where ns in [count, 2*count) is the FSE "next state
// number" of that cell.  nbBits = log - highbit(ns) and newState = (ns << nbBits) - size follow from
// it, so a block's three tables take 2.5 KB and 32 blocks (one per lane) fit one warp's 80 KB of
// shared memory, interleaved by lane (stride 32) so that the lanes' halfwords share words pairwise.
struct Tab16 {
    uint16_t* p;
    uint32_t stride;
    PNA_HD uint32_t get(uint32_t i) const { return p[i * stride]; }
    PNA_HD void set(uint32_t i, uint32_t v) const { p[i * stride] = (uint16_t)v; }
    // the same table indexed by state + size, the form in which (ns << nbBits) + bits leaves the state
    PNA_HD Tab16 by_state_plus(uint32_t size) const { return Tab16{p - (size_t)size * stride, stride}; }
};
constexpr uint32_t TAB16_LL = 0, TAB16_ML = 512, TAB16_OF = 1024, TAB16_TOTAL = 1280;

PNA_HD void fse_build_tab16(const Tab16& t, const int16_t* norm, int n_sym, int log, uint16_t* next_of) {
    const int size = 1 << log;
    int high = size - 1;
    for (int s = 0; s < n_sym; s++) {
        if (norm[s] == -1) { t.set((uint32_t)high--, (uint32_t)s << 10); next_of[s] = 1; }
        else next_of[s] = (uint16_t)norm[s];
    }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < n_sym; s++) {
        for (int i = 0; i < norm[s]; i++) {
            t.set((uint32_t)pos, (uint32_t)s << 10);
            pos = (pos + step) & mask;
            while (pos > high) pos = (pos + step) & mask;
        }
    }
    for (int u = 0; u < size; u++) {
        uint32_t s = t.get((uint32_t)u) >> 10;
        uint32_t ns = next_of[s]++;
        t.set((uint32_t)u, (s << 10) | ns);
    }
}
// kind: 0 LL, 1 OF, 2 ML.  Returns the accuracy log or -1.
PNA_HD int seq_tab16_for(const uint8_t* comp, const ZBlock* blocks, const ZBlock& b, int kind, const Tab16& t,
                         int16_t* norm, uint16_t* next_of) {
    const int max_sym = kind == 0 ? LL_MAXSYM : kind == 1 ? OF_MAXSYM : ML_MAXSYM;
    const int max_log = kind == 0 ? LL_LOG_MAX : kind == 1 ? OF_LOG_MAX : ML_LOG_MAX;
    int src = b.tsrc[kind];
    if (src < 0) {
        int log = kind == 1 ? 5 : 6;
        int n = kind == 0 ? 36 : kind == 1 ? 29 : 53;
        for (int s = 0; s < n; s++) norm[s] = (int16_t)predef_norm(kind, s);
        fse_build_tab16(t, norm, n, log, next_of);
        return log;
    }
    const ZBlock& sb = blocks[src];
    const uint8_t* d = comp + sb.src + sb.desc[kind];
    uint32_t avail = sb.size - sb.desc[kind];
    if (sb.mode[kind] == SM_RLE) {
        if (avail < 1 || d[0] > max_sym) return -1;
        t.set(0, ((uint32_t)d[0] << 10) | 1u);   // ns = 1: nbBits 0, newState 0
        return 0;
    }
    int log = 0, n_sym = 0;
    if (fse_read_ncount(d, avail, max_sym, max_log, norm, &log, &n_sym) < 0) return -1;
    fse_build_tab16(t, norm, n_sym, log, next_of);
    return log;
}
// code -> baseline | extra-bit count << 24: what decode_sequences16 expects in its llb / mlb tables (one shared-memory
// load per code gives both; the bit position depends on the count)
// extra-bit counts from the code alone
PNA_HD uint32_t ll_xbits(uint32_t c) {
    return c < 16 ? 0u : c >= 25 ? c - 19u : (uint32_t)((0x433221111ull >> (4 * (c - 16))) & 15u);
}
PNA_HD uint32_t ml_xbits(uint32_t c) {
    return c < 32 ? 0u : c >= 43 ? c - 36u : (uint32_t)((0x54433221111ull >> (4 * (c - 32))) & 15u);
}
PNA_HD uint32_t seq_pack_ll(uint32_t c) { return ll_base((int)c) | (ll_xbits(c) << 24); }
PNA_HD uint32_t seq_pack_ml(uint32_t c) { return ml_base((int)c) | (ml_xbits(c) << 24); }

// Backward bit window: 64 bits held left-aligned in a register, refilled 32 bits at a time from the
// aligned word below (prefetched one refill ahead, so the load latency is off the decode chain).
// `remain` counts the unread bits of the stream; it only ever decreases, so one check at the end
// (== 0 for sequences, >= 0 for Huffman) is equivalent to libzstd's per-step over-read checks.
struct BitWin {
    const uint32_t* words;
    uint64_t w;
    int32_t cnt;      // valid bits in w
    int64_t wp;       // index of the prefetched word
    uint32_t nx;      // words[wp]
    int64_t remain;
    PNA_HD bool init(const uint32_t* wd, const uint8_t* bytes, uint64_t begin, uint64_t len) {
        words = wd;
        w = 0; cnt = 0; wp = 0; nx = 0; remain = 0;
        if (len == 0) return false;
        const uint8_t last = bytes[begin + len - 1];
        if (last == 0) return false;
        remain = (int64_t)(len - 1) * 8 + highbit32(last);
        const uint64_t top = begin * 8 + (uint64_t)remain - 1;   // absolute index of the first bit to read
        const int64_t wi = (int64_t)(top >> 5);
        const uint32_t sh = 31u - (uint32_t)(top & 31);
        const uint64_t hi = wd[wi], lo = wi >= 1 ? wd[wi - 1] : 0u;
        w = ((hi << 32) | lo) << sh;
        cnt = 64 - (int32_t)sh;
        wp = wi - 2;
        nx = wp >= 0 ? wd[wp] : 0u;
        return true;
    }
    PNA_HD void refill() {   // afterwards cnt >= 33
        if (cnt <= 32) {
            w |= (uint64_t)nx << (32 - cnt);
            cnt += 32;
            wp--;
            nx = wp >= 0 ? words[wp] : 0u;
#if defined(__CUDA_ARCH__)
            if (wp >= 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(words + wp - 32));
#endif
        }
    }
    PNA_HD uint32_t take(uint32_t n) {   // 0 <= n <= 32, n <= cnt
        const uint32_t v = (uint32_t)((w >> 1) >> (63 - n));
        w <<= n;
        cnt -= (int32_t)n;
        remain -= n;
        return v;
    }
    PNA_HD uint32_t peek(uint32_t n) const { return (uint32_t)((w >> 1) >> (63 - n)); }   // 1 <= n <= 32
    PNA_HD void skip(uint32_t n) { w <<= n; cnt -= (int32_t)n; remain -= n; }
};

// One sequence record as the LZ stage reads it: x = offset (absolute, or symbolic REP_SYM form),
// y = min(ll, 0xFFFF) | min(ml, 0xFFFF) << 16; values >= 0xFFFF are listed in the block's escapes.
struct SeqRec { uint32_t x, y; };
constexpr uint32_t SEQ_ESC = 0xFFFFu;
constexpr int SEQ_ESC_MAX = 4;

// 64 stream bits ending just below bit `pos` (pos = number of unread bits), left-aligned: the next
// bit to read is bit 63.  wb = aligned word holding the stream's first byte, b0 = bit offset of that
// byte inside it.  Three aligned loads (independent, L1-resident) + two funnel shifts; positions
// below the stream start read the bytes in front of it (>= 11 bytes of frame/block headers, so the
// two words below wb exist) and are rejected by the final pos == 0 check.
PNA_HD uint64_t bits_window(const uint32_t* wb, uint32_t b0, int32_t pos) {
    const int32_t top = (int32_t)b0 + pos - 1;          // relative index of the first bit to read (>= -1)
    const int32_t wi = top >> 5;                        // arithmetic shift: -1 -> word -1
    const uint32_t sh = 31u - ((uint32_t)top & 31u);
    const uint32_t h = wb[wi], m = wb[wi - 1], l = wb[wi - 2];
#if defined(__CUDA_ARCH__)
    const uint32_t whi = __funnelshift_l(m, h, sh), wlo = __funnelshift_l(l, m, sh);
#else
    const uint32_t whi = sh ? (h << sh) | (m >> (32 - sh)) : h, wlo = sh ? (m << sh) | (l >> (32 - sh)) : m;
#endif
    return ((uint64_t)whi << 32) | wlo;
}
// The high word of (hi:lo) << n, 0 <= n <= 31: hi shifted up by n with the top n bits of lo below it.  One SHF on the
// GPU.  The sequence loop cuts every field with it: (prefix:window) << n appends the window's next n bits to prefix.
PNA_HD uint32_t shl_hi(uint32_t lo, uint32_t hi, uint32_t n) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, n);
#else
    return (uint32_t)(((((uint64_t)hi << 32) | lo) << n) >> 32);
#endif
}

// Sequence decode of one block by ONE thread (a lane of zstd_seq_kernel).  Position-based bit
// reader: per sequence one 64-bit window is fetched at the current bit position while the three
// table cells are looked up; all fields of the sequence (<= 64 bits in every stream the reference
// writes; longer ones take a second window) are cut out of it, and only
//   state -> table cell -> bit counts -> next position / next state
// is loop-carried.  Errors are collected in a flag (no early exits inside the loop).
// llb/mlb: by code, value baseline | extra-bit count << 24 (seq_pack_ll / seq_pack_ml).  Same accept/reject behaviour as decode_sequences().
// Where decode_sequences16 takes its 64-bit windows from.  GlobalBitSrc: straight from the arena (three aligned loads
// per window, the sector 128 bytes below pulled into L1 ahead of use); zstd_seq_kernel uses a per-lane shared-memory
// ring fed by cp.async instead (kernels_zstd.cuh: RingBitSrc), which takes the HBM/L2 latency off the decode chain.
struct GlobalBitSrc {
    const uint32_t* words;
    const uint32_t* wb;
    uint32_t b0;
    PNA_HD void init(const uint32_t* w, uint64_t begin, int32_t /*pos*/) { words = w; wb = w + (begin >> 2); b0 = (uint32_t)(begin & 3) * 8; }
    PNA_HD uint64_t window(int32_t pos) {
#if defined(__CUDA_ARCH__)
        const uint32_t* pf = wb + (((int32_t)b0 + pos) >> 5) - 32;
        asm volatile("prefetch.global.L1 [%0];" ::"l"(pf < words ? words : pf));
#endif
        return bits_window(wb, b0, pos);
    }
};

// One block's sequence stream as a stepper.  A step is cut in three phases:
//   advance(i)  the loop-carried part: cells -> bit counts -> fields of this sequence, next position, next states
//   fetch()     the NEXT sequence's bit window and table cells are requested
//   emit(i)     this sequence's values, repeat-offset logic and the store, in the latency shadow of those loads
// States are kept as FSE state + table size, which is what (ns << nbBits) + bits gives; the tables are addressed through
// Tab16::by_state_plus.  Every field is cut from the top of the window with one funnel shift (shl_hi).
template <class Src>
struct SeqStream {
    Src src;
    Tab16 tll, tof, tml;
    const uint32_t *llb, *mlb;
    SeqRec* out;
    uint32_t ulll, ulof, ulml, nseq, lit_regen;
    uint32_t sll, sof, sml, ell, eof, eml;
    int32_t pos;       // unread bits; below 0 once the stream is over-read (windows are then read at 0), so end() checks == 0
    uint64_t W;
    uint32_t rep0, rep1, rep2, lit_sum, match_sum, ne, err;
    // The two per-sequence error tests of the repeat-offset logic, as extremes that end() tests once:
    //   omin == 0           "rep0 - 1" of an absolute rep0 == 1.  No other offset can be 0, and a symbolic "rep0 - 1"
    //                       (delta + 1) cannot carry into the slot bits: delta <= nseq < 2^17.
    //   omax > 2^31 + 2     a new offset (ofv > 3) of 2^31 or more, beyond any legal window.
    uint32_t omin, omax;
    ZBlock* blk;   // the block's record: escapes (rare) and results go straight there -- the struct holds scalars only, so that
                   // a lane's streams live in registers (an array member would pin them to local memory, which the sequence
                   // kernel's shared-memory carve-out leaves without L1)
    // fields of the sequence between advance() and emit()
    uint32_t f_ofv, f_mlx, f_llx, f_pll, f_pml;

    // everything in front of the loop; ST_OK or the status the block fails with
    PNA_HD int32_t begin(const uint32_t* words, const uint8_t* comp, ZBlock& b, const Tab16& tll_, const Tab16& tof_, const Tab16& tml_,
                         int lll, int lof, int lml, const uint32_t* llb_, const uint32_t* mlb_, SeqRec* out_) {
        llb = llb_; mlb = mlb_; out = out_; blk = &b;
        const uint64_t begin_at = b.src + b.bs_pos;
        const uint32_t len = b.bs_len;
        nseq = b.nseq; lit_regen = b.lit_regen;
        if (len == 0) return ST_INVALID_DATA;
        const uint8_t last = comp[begin_at + len - 1];
        if (last == 0) return ST_INVALID_DATA;
        pos = (int32_t)(len - 1) * 8 + highbit32(last);
        ulll = (uint32_t)lll; ulof = (uint32_t)lof; ulml = (uint32_t)lml;
        if (pos < (int32_t)(ulll + ulof + ulml)) return ST_INVALID_DATA;
        tll = tll_.by_state_plus(1u << lll); tof = tof_.by_state_plus(1u << lof); tml = tml_.by_state_plus(1u << lml);
        src.init(words, begin_at, pos);
        W = src.window(pos);
        uint32_t h = (uint32_t)(W >> 32);   // the initial states, <= 9 + 8 + 9 bits: 1 << log prefixes the state's bits
        sll = shl_hi(h, 1u, ulll); h <<= ulll;
        sof = shl_hi(h, 1u, ulof); h <<= ulof;
        sml = shl_hi(h, 1u, ulml);
        pos -= (int32_t)(ulll + ulof + ulml);
        rep0 = REP_SYM | (0u << 29); rep1 = REP_SYM | (1u << 29); rep2 = REP_SYM | (2u << 29);
        lit_sum = 0; match_sum = 0;            // < 2^32: nseq < 2^17 values < 2^17 each
        ne = 0; err = 0; omin = 0xFFFFFFFFu; omax = 0;
        W = src.window(pos);
        ell = tll.get(sll); eof = tof.get(sof); eml = tml.get(sml);
        return ST_OK;
    }
    PNA_HD void advance(uint32_t i) {
        const uint32_t cof = eof >> 10;
        const uint32_t pll = llb[ell >> 10], pml = mlb[eml >> 10];   // baseline | extra bits << 24 (seq_pack_ll / _ml)
        const uint32_t xll = pll >> 24, xml = pml >> 24;
        const uint32_t nsl = ell & 1023u, nsm = eml & 1023u, nso = eof & 1023u;
        const uint32_t nbl = ulll - (uint32_t)highbit32(nsl), nbm = ulml - (uint32_t)highbit32(nsm),
                       nbo = ulof - (uint32_t)highbit32(nso);
        const uint32_t xb = cof + xml + xll;                 // value bits: offset, match length, literal length
        const uint32_t nbs = i + 1 < nseq ? nbl + nbm + nbo : 0u;   // the last sequence reads no state bits
        // cut from the top: (h:l) is the window, shifted up past each field as it is taken
        uint32_t h = (uint32_t)(W >> 32), l = (uint32_t)W;
        f_ofv = shl_hi(h, 1u, cof);                          // (1 << cof) + cof extra bits
        h = shl_hi(l, h, cof); l <<= cof;
        f_mlx = shl_hi(h, 0u, xml);
        h = shl_hi(l, h, xml); l <<= xml;
        f_llx = shl_hi(h, 0u, xll);
        h = shl_hi(l, h, xll);
        if (xb + nbs > 64u) {   // > 64 bits in one sequence (offset codes > 22 with long length codes): second window for the states
            const int32_t p2 = pos - (int32_t)xb;
            h = p2 >= 0 ? (uint32_t)(src.window(p2) >> 32) : 0u;
        }
        // next states (ns << nb) + nb bits, in the order LL, ML, OF; the last sequence's are never used
        sll = shl_hi(h, nsl, nbl); h <<= nbl;
        sml = shl_hi(h, nsm, nbm); h <<= nbm;
        sof = shl_hi(h, nso, nbo);
        pos -= (int32_t)(xb + nbs);
        f_pll = pll; f_pml = pml;
    }
    PNA_HD void fetch() {
        W = src.window(pos < 0 ? 0 : pos);                   // keep the reads inside the arena on corrupt input
        ell = tll.get(sll); eof = tof.get(sof); eml = tml.get(sml);
    }
    PNA_HD void emit(uint32_t i) {
        const uint32_t ml = (f_pml & 0xFFFFFFu) + f_mlx;
        const uint32_t ll = (f_pll & 0xFFFFFFu) + f_llx;
        const uint32_t ofv = f_ofv;
        // repeat-offset logic (RFC 8878 3.1.1.5), branch-free; offsets may be symbolic (REP_SYM) in the block's incoming history.
        // idx 0..2 picks rep0..rep2; idx >= 3 is a new offset (ofv > 3) or "rep0 - 1" (ofv == 3 with ll == 0)
        const uint32_t idx = ofv - (ll < 1u ? ll : 1u);
        const uint32_t dec = rep0 - 1u + ((rep0 >> 30) & 2u);     // "rep0 - 1" (symbolic: delta + 1)
        const uint32_t nw = ofv == 3u ? dec : ofv - 3u;
        const uint32_t r12 = idx >= 2u ? rep2 : rep1;
        const uint32_t off = idx >= 3u ? nw : idx >= 1u ? r12 : rep0;
        omin = off < omin ? off : omin;
        omax = ofv > omax ? ofv : omax;
        rep2 = idx >= 2u ? rep1 : rep2;
        rep1 = idx >= 1u ? rep0 : rep1;
        rep0 = off;
        SeqRec r;
        r.x = off;
        r.y = ll + (ml << 16);
        if ((ll | ml) >= SEQ_ESC) {                          // cheap superset of "a length does not fit 16 bits" (rare)
            if (ll >= SEQ_ESC || ml >= SEQ_ESC) {
                if (ne < (uint32_t)SEQ_ESC_MAX) { blk->esc_idx[ne] = i; blk->esc_ll[ne] = ll; blk->esc_ml[ne] = ml; }
                else err |= 1u;                              // > 4 such sequences cannot fit a 128 KiB block
                ne++;
            }
            r.y = (ll < SEQ_ESC ? ll : SEQ_ESC) | ((ml < SEQ_ESC ? ml : SEQ_ESC) << 16);
        }
#if defined(__CUDA_ARCH__)
        *reinterpret_cast<uint2*>(out++) = make_uint2(r.x, r.y);   // one 8-byte store (records are 8-byte aligned)
#else
        *out++ = r;
#endif
        lit_sum += ll; match_sum += ml;
    }
    PNA_HD void step(uint32_t i) { advance(i); fetch(); emit(i); }
    // after the last sequence: final checks, block totals, outgoing history, escapes
    PNA_HD int32_t end() {
        if (err || pos != 0 || omin == 0 || omax > 0x80000002u) return ST_INVALID_DATA;
        if (lit_sum > lit_regen) return ST_INVALID_DATA;
        const uint64_t outsz = (uint64_t)lit_regen + match_sum;
        if (outsz > BLOCK_MAX) return ST_INVALID_DATA;
        ZBlock& b = *blk;
        b.out_size = (uint32_t)outsz;
        b.lit_used = lit_sum;
        b.rep_out[0] = rep0; b.rep_out[1] = rep1; b.rep_out[2] = rep2;
        b.esc_n = ne;
        return ST_OK;
    }
};

template <class Src>
PNA_HD int32_t decode_sequences16_from(Src& src, const uint32_t* words, const uint8_t* comp, ZBlock& b, const Tab16& tll,
                                       const Tab16& tof, const Tab16& tml, int lll, int lof, int lml,
                                       const uint32_t* llb, const uint32_t* mlb, SeqRec* out, uint32_t* esc_n,
                                       uint32_t* esc_idx, uint32_t* esc_ll, uint32_t* esc_ml) {
    SeqStream<Src> st;
    st.src = src;
    const int32_t rc = st.begin(words, comp, b, tll, tof, tml, lll, lof, lml, llb, mlb, out);
    if (rc != ST_OK) return rc;
    for (uint32_t i = 0; i < st.nseq; i++) st.step(i);
    const int32_t rc2 = st.end();
    if (rc2 == ST_OK) {
        *esc_n = b.esc_n;
        for (uint32_t q = 0; q < b.esc_n && q < (uint32_t)SEQ_ESC_MAX; q++) { esc_idx[q] = b.esc_idx[q]; esc_ll[q] = b.esc_ll[q]; esc_ml[q] = b.esc_ml[q]; }
    }
    return rc2;
}
PNA_HD int32_t decode_sequences16(const uint32_t* words, const uint8_t* comp, ZBlock& b, const Tab16& tll,
                                  const Tab16& tof, const Tab16& tml, int lll, int lof, int lml,
                                  const uint32_t* llb, const uint32_t* mlb, SeqRec* out, uint32_t* esc_n,
                                  uint32_t* esc_idx, uint32_t* esc_ll, uint32_t* esc_ml) {
    GlobalBitSrc src;
    return decode_sequences16_from(src, words, comp, b, tll, tof, tml, lll, lof, lml, llb, mlb, out, esc_n, esc_idx, esc_ll, esc_ml);
}

// ---------------------------------------------------------------------------------------------
// Huffman tree description -> single-symbol decode table (libzstd HUF_readStats + HUF_readDTableX1).
// table: uint16_t[1<<log] entries (sym | nbBits<<8).  weights: uint8_t[256] scratch.  fse: FseEntry[64] scratch.
// Returns header bytes consumed (>0) or -1; *table_log receives the log.
PNA_HD int huf_read_table(const uint32_t* words, const uint8_t* comp, uint64_t at, uint32_t avail, uint16_t* table,
                          int* table_log, uint8_t* weights, FseEntry* fse) {
    if (avail < 1) return -1;
    const uint8_t* p = comp + at;
    uint32_t isize = p[0];
    uint32_t n_w = 0;
    if (isize >= 128) {
        n_w = isize - 127;
        isize = (n_w + 1) / 2;
        if (isize + 1 > avail) return -1;
        for (uint32_t n = 0; n < n_w; n += 2) {
            weights[n] = p[1 + n / 2] >> 4;
            weights[n + 1] = p[1 + n / 2] & 15;
        }
    } else {
        if (isize + 1 > avail || isize == 0) return -1;
        int16_t norm[256];
        int log = 0, n_sym = 0;
        int hdr = fse_read_ncount(p + 1, isize, 255, 6, norm, &log, &n_sym);
        if (hdr < 0) return -1;
        // plain FSE decode table (FSE_buildDTable)
        const int size = 1 << log;
        uint16_t next_of[256];
        int high = size - 1;
        for (int s = 0; s < n_sym; s++) {
            if (norm[s] == -1) { fse[high--].sym = (uint8_t)s; next_of[s] = 1; }
            else next_of[s] = (uint16_t)norm[s];
        }
        const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
        int pos = 0;
        for (int s = 0; s < n_sym; s++)
            for (int i = 0; i < norm[s]; i++) {
                fse[pos].sym = (uint8_t)s;
                pos = (pos + step) & mask;
                while (pos > high) pos = (pos + step) & mask;
            }
        for (int u = 0; u < size; u++) {
            uint32_t ns = next_of[fse[u].sym]++;
            int nb = log - highbit32(ns);
            fse[u].nb = (uint8_t)nb;
            fse[u].next = (uint16_t)((ns << nb) - (uint32_t)size);
        }
        // two interleaved states, FSE_decompress_usingDTable tail semantics
        BackBits bb;
        if ((uint32_t)hdr >= isize) return -1;
        if (!bb.init(words, comp, at + 1 + (uint32_t)hdr, isize - (uint32_t)hdr)) return -1;
        uint32_t s1 = bb.read(log), s2 = bb.read(log);
        if (bb.pos < 0) return -1;
        for (;;) {
            if (n_w > 253) return -1;
            weights[n_w++] = fse[s1].sym;
            s1 = fse[s1].next + bb.read(fse[s1].nb);
            if (bb.pos < 0) { weights[n_w++] = fse[s2].sym; break; }
            if (n_w > 253) return -1;
            weights[n_w++] = fse[s2].sym;
            s2 = fse[s2].next + bb.read(fse[s2].nb);
            if (bb.pos < 0) { weights[n_w++] = fse[s1].sym; break; }
        }
    }
    if (n_w == 0 || n_w > 255) return -1;
    uint32_t rank[HUF_LOG_MAX + 2];
    for (int i = 0; i < HUF_LOG_MAX + 2; i++) rank[i] = 0;
    uint32_t total = 0;
    for (uint32_t n = 0; n < n_w; n++) {
        if (weights[n] > HUF_LOG_MAX) return -1;
        rank[weights[n]]++;
        total += (1u << weights[n]) >> 1;
    }
    if (total == 0) return -1;
    int log = highbit32(total) + 1;
    if (log > HUF_LOG_MAX) return -1;
    uint32_t rest = (1u << log) - total;
    int last_w = highbit32(rest) + 1;
    if ((1u << (last_w - 1)) != rest) return -1;   // must be a clean power of two
    weights[n_w] = (uint8_t)last_w;
    rank[last_w]++;
    if (rank[1] < 2 || (rank[1] & 1)) return -1;
    // rank start positions, lowest weight (longest code) first
    uint32_t start[HUF_LOG_MAX + 2];
    uint32_t nxt = 0;
    for (int w = 1; w <= log; w++) { start[w] = nxt; nxt += rank[w] << (w - 1); }
    for (uint32_t s = 0; s <= n_w; s++) {
        uint32_t w = weights[s];
        if (!w) continue;
        uint32_t len = (1u << w) >> 1;
        uint16_t e = (uint16_t)(s | ((uint32_t)(log + 1 - (int)w) << 8));
        for (uint32_t u = 0; u < len; u++) table[start[w] + u] = e;
        start[w] += len;
    }
    *table_log = log;
    return (int)isize + 1;
}

// Decode one Huffman stream of `count` symbols.  Returns false on corruption.
PNA_HD bool huf_decode_stream(const uint32_t* words, const uint8_t* comp, uint64_t begin, uint32_t len,
                              const uint16_t* table, int log, uint8_t* dst, uint32_t count) {
    BackBits bb;
    if (!bb.init(words, comp, begin, len)) return false;
    for (uint32_t i = 0; i < count; i++) {
        uint16_t e = table[bb.peek_top(log)];
        dst[i] = (uint8_t)e;
        bb.pos -= (e >> 8);
        if (bb.pos < 0) return false;
    }
    // libzstd >= 1.5.4's fast Huffman loops validate the produced length only, not that every bit of
    // the stream was consumed; leftover bits are therefore accepted, an over-read is not.
    return true;
}

// Same stream decode on the register bit window (kernels_zstd.cuh zstd_lit_kernel): two symbols per
// refill, output gathered into aligned 32-bit stores.  Table stride lets 4 lanes share one table.
PNA_HD bool huf_decode_stream_w(const uint32_t* words, const uint8_t* comp, uint64_t begin, uint32_t len,
                                const uint16_t* table, int log, uint8_t* dst, uint32_t count) {
    BitWin bw;
    if (!bw.init(words, comp, begin, len)) return false;
    const uint32_t ulog = (uint32_t)log;
    uint32_t i = 0;
#define PNA_HUF_SYM(var_) do { const uint32_t e__ = table[bw.peek(ulog)]; var_ = e__ & 0xFFu; bw.skip(e__ >> 8); } while (0)
    // head: bytes until dst is 4-byte aligned
    while (i < count && (((uintptr_t)(dst + i)) & 3) != 0) {
        bw.refill();
        uint32_t s; PNA_HUF_SYM(s);
        dst[i++] = (uint8_t)s;
    }
    for (; i + 4 <= count; i += 4) {
        uint32_t s0, s1, s2, s3;
        bw.refill(); PNA_HUF_SYM(s0); PNA_HUF_SYM(s1);
        bw.refill(); PNA_HUF_SYM(s2); PNA_HUF_SYM(s3);
        *reinterpret_cast<uint32_t*>(dst + i) = s0 | (s1 << 8) | (s2 << 16) | (s3 << 24);
    }
    for (; i < count; i++) {
        bw.refill();
        uint32_t s; PNA_HUF_SYM(s);
        dst[i] = (uint8_t)s;
    }
#undef PNA_HUF_SYM
    return bw.remain >= 0;   // leftover bits are accepted (libzstd >= 1.5.4 fast loops), an over-read is not
}

// ---------------------------------------------------------------------------------------------
// Frame scan.  Walks the frames and block headers of one entry's compressed stream.  When `blocks`
// is null only counts.  Returns the entry status; *n_blocks = number of blocks found.
// One block header as the frame walk records it: the walk is the only inherently serial step (a block's position is
// known only after every block header in front of it was read), so it writes 16 bytes per block and leaves building the
// 200-byte ZBlock records to a thread per block (zstd_fill_kernel).
struct WalkRec {
    uint64_t src;       // byte offset of the block content inside the comp arena
    uint32_t entry;
    uint32_t bits;      // size (bits 0-20) | type << 21 | first_in_frame << 23
};
PNA_HD void zblock_from_walk(const WalkRec& w, ZBlock& z) {
    memset(&z, 0, sizeof z);
    z.src = w.src;
    z.entry = w.entry;
    z.size = w.bits & 0x1FFFFFu;
    z.type = (uint8_t)((w.bits >> 21) & 3u);
    z.first_in_frame = (uint8_t)((w.bits >> 23) & 1u);
    z.out_size = z.type == BT_COMPRESSED ? 0 : z.size;
    z.tsrc[0] = z.tsrc[1] = z.tsrc[2] = -1;
    z.huf_src = -1;
}
PNA_HD int32_t scan_entry(const uint8_t* comp, uint64_t base, uint64_t len, uint32_t entry, ZBlock* blocks,
                          uint32_t* n_blocks, WalkRec* walk = nullptr, uint32_t walk_cap = 0) {
    uint64_t pos = 0;
    uint32_t nb = 0;
    int32_t st = ST_OK;
    while (pos < len) {
        if (len - pos < 4) { st = ST_UNEXPECTED_EOF; break; }
        uint32_t magic = load_le32(comp + base + pos);
        if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {  // skippable frame
            if (len - pos < 8) { st = ST_UNEXPECTED_EOF; break; }
            uint64_t sz = load_le32(comp + base + pos + 4);
            if (len - pos - 8 < sz) { st = ST_UNEXPECTED_EOF; break; }
            pos += 8 + sz;
            continue;
        }
        if (magic != MAGIC) { st = ST_INVALID_DATA; break; }
        if (len - pos < 5) { st = ST_UNEXPECTED_EOF; break; }
        uint8_t fhd = comp[base + pos + 4];
        uint32_t fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, checksum = (fhd >> 2) & 1, did_flag = fhd & 3;
        if (fhd & 0x08) { st = ST_INVALID_DATA; break; }  // reserved bit
        uint32_t did_size = did_flag == 3 ? 4 : did_flag;
        uint32_t fcs_size = fcs_flag == 0 ? single : (1u << fcs_flag);
        uint32_t hdr = 5 + (single ? 0 : 1) + did_size + fcs_size;
        if (len - pos < hdr) { st = ST_UNEXPECTED_EOF; break; }
        const uint8_t* h = comp + base + pos + 5;
        uint64_t window = 0;
        if (!single) {
            uint8_t wd = *h++;
            uint32_t wlog = 10 + (wd >> 3);
            if (wlog > 30) { st = ST_INVALID_DATA; break; }
            window = (1ull << wlog) + ((1ull << wlog) >> 3) * (wd & 7);
        }
        uint32_t dict_id = 0;
        for (uint32_t i = 0; i < did_size; i++) dict_id |= (uint32_t)h[i] << (8 * i);
        h += did_size;
        if (dict_id != 0) { st = ST_INVALID_DATA; break; }  // no dictionary is ever supplied: libzstd dictionary_wrong
        uint64_t fcs = 0;
        for (uint32_t i = 0; i < fcs_size; i++) fcs |= (uint64_t)h[i] << (8 * i);
        if (fcs_size == 2) fcs += 256;
        if (single) window = fcs;
        if (window > WINDOW_MAX) { st = ST_INVALID_DATA; break; }  // frameParameter_windowTooLarge
        uint64_t block_max = window < BLOCK_MAX ? window : BLOCK_MAX;
        pos += hdr;
        bool first = true, done = false;
        while (!done) {
            if (len - pos < 3) { st = ST_UNEXPECTED_EOF; break; }
            uint32_t bh = load_le24(comp + base + pos);
            uint32_t last = bh & 1, type = (bh >> 1) & 3, size = bh >> 3;
            if (type == 3) { st = ST_INVALID_DATA; break; }
            if (size > block_max) { st = ST_INVALID_DATA; break; }
            uint64_t content = type == BT_RLE ? 1 : size;
            if (len - pos - 3 < content) { st = ST_UNEXPECTED_EOF; break; }
            if (blocks) {
                ZBlock z;
                memset(&z, 0, sizeof z);
                z.src = base + pos + 3;
                z.entry = entry;
                z.size = size;
                z.type = (uint8_t)type;
                z.first_in_frame = first ? 1 : 0;
                z.out_size = type == BT_COMPRESSED ? 0 : size;
                z.tsrc[0] = z.tsrc[1] = z.tsrc[2] = -1;
                z.huf_src = -1;
                blocks[nb] = z;
            }
            if (walk && nb < walk_cap) walk[nb] = WalkRec{base + pos + 3, entry, size | (type << 21) | ((first ? 1u : 0u) << 23)};
            nb++;
            first = false;
            pos += 3 + content;
            if (last) {
                if (checksum) {
                    if (len - pos < 4) { st = ST_UNEXPECTED_EOF; break; }
                    pos += 4;  // XXH64 low 32 bits: not verified here (reference-written frames carry none)
                }
                done = true;
            }
        }
        if (st != ST_OK) break;
    }
    *n_blocks = nb;
    return st;
}

// Parse the inside of one compressed block: literal section header, sequence header, table
// description offsets.  Fills the ZBlock fields; returns status.
PNA_HD int32_t parse_block(const uint8_t* comp, ZBlock& b) {
    if (b.type != BT_COMPRESSED) return ST_OK;
    const uint8_t* p = comp + b.src;
    const uint32_t n = b.size;
    if (n < 2) return ST_INVALID_DATA;
    uint8_t b0 = p[0];
    uint32_t lt = b0 & 3, fmt = (b0 >> 2) & 3;
    uint32_t lh = 0, regen = 0, csize = 0, streams = 1;
    if (lt == LT_COMPRESSED || lt == LT_TREELESS) {
        if (n < 5) return ST_INVALID_DATA;
        uint32_t lhc = load_le32(p);
        if (fmt < 2) { streams = fmt ? 4 : 1; lh = 3; regen = (lhc >> 4) & 0x3FF; csize = (lhc >> 14) & 0x3FF; }
        else if (fmt == 2) { streams = 4; lh = 4; regen = (lhc >> 4) & 0x3FFF; csize = lhc >> 18; }
        else { streams = 4; lh = 5; regen = (lhc >> 4) & 0x3FFFF; csize = (lhc >> 22) + ((uint32_t)p[4] << 10); }
        if (regen > BLOCK_MAX) return ST_INVALID_DATA;
        if (streams == 4 && regen < 6) return ST_INVALID_DATA;
        if (csize + lh > n) return ST_INVALID_DATA;
    } else {
        if (fmt == 0 || fmt == 2) { lh = 1; regen = b0 >> 3; }
        else if (fmt == 1) { lh = 2; regen = load_le16(p) >> 4; }
        else { if (n < 3) return ST_INVALID_DATA; lh = 3; regen = load_le24(p) >> 4; }
        if (regen > BLOCK_MAX) return ST_INVALID_DATA;
        csize = lt == LT_RAW ? regen : 1;
        if (csize + lh > n) return ST_INVALID_DATA;
    }
    b.lit_type = (uint8_t)lt;
    b.lit_streams = (uint8_t)streams;
    b.lit_regen = regen;
    b.lit_csize = csize;
    b.lit_pos = lh;
    // sequences section
    uint32_t ip = lh + csize;
    if (ip >= n) return ST_INVALID_DATA;
    uint32_t nseq = p[ip++];
    if (nseq > 0x7F) {
        if (nseq == 0xFF) {
            if (ip + 2 > n) return ST_INVALID_DATA;
            nseq = load_le16(p + ip) + 0x7F00;
            ip += 2;
        } else {
            if (ip >= n) return ST_INVALID_DATA;
            nseq = ((nseq - 0x80) << 8) + p[ip++];
        }
    }
    b.nseq = nseq;
    if (nseq == 0) {
        if (ip != n) return ST_INVALID_DATA;
        b.out_size = regen;
        return ST_OK;
    }
    if (ip + 1 > n) return ST_INVALID_DATA;
    uint8_t modes = p[ip++];
    if (modes & 3) return ST_INVALID_DATA;
    b.mode[0] = modes >> 6; b.mode[1] = (modes >> 4) & 3; b.mode[2] = (modes >> 2) & 3;
    b.seq_pos = ip;
    for (int k = 0; k < 3; k++) {
        const int max_sym = k == 0 ? LL_MAXSYM : k == 1 ? OF_MAXSYM : ML_MAXSYM;
        const int max_log = k == 0 ? LL_LOG_MAX : k == 1 ? OF_LOG_MAX : ML_LOG_MAX;
        b.desc[k] = ip;
        if (b.mode[k] == SM_RLE) {
            if (ip >= n || p[ip] > max_sym) return ST_INVALID_DATA;
            ip += 1;
        } else if (b.mode[k] == SM_FSE) {
            int16_t norm[64];
            int log = 0, ns = 0;
            int used = fse_read_ncount(p + ip, n - ip, max_sym, max_log, norm, &log, &ns);
            if (used < 0) return ST_INVALID_DATA;
            ip += (uint32_t)used;
        }
    }
    if (ip >= n) return ST_INVALID_DATA;
    b.bs_pos = ip;
    b.bs_len = n - ip;
    return ST_OK;
}

// Resolve Repeat_Mode / treeless sources for the blocks [first, first+count) of ONE entry, in order.
PNA_HD int32_t resolve_sources(ZBlock* blocks, uint32_t first, uint32_t count) {
    int32_t cur[3] = {-2, -2, -2};  // -2 = nothing usable yet (start of frame)
    int32_t huf = -2;
    for (uint32_t i = first; i < first + count; i++) {
        ZBlock& b = blocks[i];
        if (b.first_in_frame) { cur[0] = cur[1] = cur[2] = -2; huf = -2; }
        if (b.type != BT_COMPRESSED || b.status != ST_OK) continue;
        if (b.lit_type == LT_COMPRESSED) huf = (int32_t)i;
        else if (b.lit_type == LT_TREELESS) { if (huf < 0) return ST_INVALID_DATA; }
        b.huf_src = huf;
        if (b.nseq == 0) continue;
        for (int k = 0; k < 3; k++) {
            if (b.mode[k] == SM_PREDEF) cur[k] = -1;
            else if (b.mode[k] == SM_REPEAT) { if (cur[k] == -2) return ST_INVALID_DATA; }
            else cur[k] = (int32_t)i;
            b.tsrc[k] = cur[k];
        }
    }
    return ST_OK;
}

// ---------------------------------------------------------------------------------------------
// Sequence decode of one block (serial; one thread).  tabs/logs for LL, OF, ML already built.
// Writes ll/ml/off triples; offsets may be symbolic (REP_SYM) in the block's incoming history.
PNA_HD int32_t decode_sequences(const uint32_t* words, const uint8_t* comp, ZBlock& b, const SeqEntry* tll,
                                const SeqEntry* tof, const SeqEntry* tml, int lll, int lof, int lml, uint32_t* o_ll,
                                uint32_t* o_ml, uint32_t* o_off) {
    BackBits bb;
    if (!bb.init(words, comp, b.src + b.bs_pos, b.bs_len)) return ST_INVALID_DATA;
    uint32_t sll = bb.read(lll), sof = bb.read(lof), sml = bb.read(lml);
    if (bb.pos < 0) return ST_INVALID_DATA;
    uint32_t rep0 = REP_SYM | (0u << 29), rep1 = REP_SYM | (1u << 29), rep2 = REP_SYM | (2u << 29);
    uint64_t lit_sum = 0, match_sum = 0;
    const uint32_t nseq = b.nseq;
    for (uint32_t i = 0; i < nseq; i++) {
        SeqEntry ell = tll[sll], eof = tof[sof], eml = tml[sml];
        uint32_t ofv = eof.base + bb.read(eof.nb_extra);
        uint32_t ml = eml.base + bb.read(eml.nb_extra);
        uint32_t ll = ell.base + bb.read(ell.nb_extra);
        uint32_t off;
        if (ofv > 3) {
            off = ofv - 3;
            if (off & REP_SYM) return ST_INVALID_DATA;  // beyond any legal window
            rep2 = rep1; rep1 = rep0; rep0 = off;
        } else {
            uint32_t idx = ofv - 1 + (ll == 0 ? 1u : 0u);
            if (idx == 0) off = rep0;
            else if (idx == 1) { off = rep1; rep1 = rep0; rep0 = off; }
            else if (idx == 2) { off = rep2; rep2 = rep1; rep1 = rep0; rep0 = off; }
            else {
                if (rep0 & REP_SYM) { off = rep0 + 1; if ((off & 0x1FFFFFFFu) == 0) return ST_INVALID_DATA; }
                else { off = rep0 - 1; if (off == 0) return ST_INVALID_DATA; }
                rep2 = rep1; rep1 = rep0; rep0 = off;
            }
        }
        o_ll[i] = ll; o_ml[i] = ml; o_off[i] = off;
        lit_sum += ll; match_sum += ml;
        if (i + 1 < nseq) {
            sll = ell.next + bb.read(ell.nb);
            sml = eml.next + bb.read(eml.nb);
            sof = eof.next + bb.read(eof.nb);
        }
        if (bb.pos < 0) return ST_INVALID_DATA;
    }
    if (bb.pos != 0) return ST_INVALID_DATA;
    if (lit_sum > b.lit_regen) return ST_INVALID_DATA;
    uint64_t out = (uint64_t)b.lit_regen + match_sum;
    if (out > BLOCK_MAX) return ST_INVALID_DATA;
    b.out_size = (uint32_t)out;
    b.lit_used = (uint32_t)lit_sum;
    b.rep_out[0] = rep0; b.rep_out[1] = rep1; b.rep_out[2] = rep2;
    return ST_OK;
}

// Per-entry prefix pass: output offsets of every block, frame starts and the absolute incoming
// repeat-offset history of each block (the outgoing one of a block is symbolic in its incoming one).
PNA_HD uint32_t resolve_rep(uint32_t v, const uint32_t rep_in[3]);
PNA_HD int32_t prefix_entry(ZBlock* blocks, uint32_t first, uint32_t count, uint64_t out_base, uint64_t* total_out) {
    uint64_t pos = 0, frame_start = 0;
    uint32_t rep[3] = {1, 4, 8};
    int32_t st = ST_OK;
    for (uint32_t i = first; i < first + count; i++) {
        ZBlock& b = blocks[i];
        if (b.first_in_frame) { rep[0] = 1; rep[1] = 4; rep[2] = 8; frame_start = pos; }
        b.out_off = out_base + pos;
        b.frame_out = out_base + frame_start;
        b.rep_in[0] = rep[0]; b.rep_in[1] = rep[1]; b.rep_in[2] = rep[2];
        if (b.status != ST_OK) { if (st == ST_OK) st = b.status; continue; }
        if (b.type == BT_COMPRESSED && b.nseq > 0) {
            uint32_t r0 = resolve_rep(b.rep_out[0], b.rep_in), r1 = resolve_rep(b.rep_out[1], b.rep_in),
                     r2 = resolve_rep(b.rep_out[2], b.rep_in);
            if (!r0 || !r1 || !r2) { b.status = ST_INVALID_DATA; if (st == ST_OK) st = ST_INVALID_DATA; continue; }
            rep[0] = r0; rep[1] = r1; rep[2] = r2;
        }
        pos += b.out_size;
    }
    *total_out = pos;
    return st;
}

// resolve a possibly symbolic offset against an absolute incoming history; 0 = corrupt
PNA_HD uint32_t resolve_rep(uint32_t v, const uint32_t rep_in[3]) {
    if (!(v & REP_SYM)) return v;
    uint32_t slot = (v >> 29) & 3, delta = v & 0x1FFFFFFFu;
    uint32_t base = rep_in[slot];
    return base > delta ? base - delta : 0;
}

}  // namespace zs
}  // namespace pna
