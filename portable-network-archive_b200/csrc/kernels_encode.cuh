// kernels_encode.cuh -- sm_100a kernels of the encode seam (K6/K7 + cipher encrypt + FDAT CRC):
//   lz_match_kernel      (warp per 32 KiB segment)  warp-synchronous greedy LZ77: 32 positions per step, candidates
//                        from a shared-memory hash table AND from the step's own lanes (__match_any_sync), greedy
//                        parse of the step by pointer doubling with shuffles, sequences + literals compacted by ballots
//   enc_block_kernel     (lane per segment)         zstd block (predefined-FSE sequences + repeat offsets, Huffman or raw literals) or deflate
//                        fixed-Huffman block, written by the PNA_HD writers of encode_core.cuh
//   enc_layout_kernel    (thread per entry)         frame header / trailer, piece list of the compressed stream, Adler-32
//   encrypt_tiles_kernel (thread per 16-byte block) gather the pieces, AES/Camellia CTR (or plain copy) into the output
//   cbc_encrypt_kernel   (lane per entry)           CBC is a serial chain per stream: entry-level parallelism only
//   crc_clip_kernel      clips the bound-based CRC tile table to the produced stream lengths (no host round trip)
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"
#include "encode_core.cuh"
#include "lzma_enc_core.cuh"
#include "kernels_crc_cipher.cuh"
#include "kernels_gcm.cuh"

namespace pna {
namespace enc {

struct SegRec {            // one segment (host fills the first group, kernels the second)
    uint64_t plain_off;    // all offsets are relative to the work arena
    uint64_t lit_off;
    uint64_t tmp_off;      // 16 bytes of head + body
    uint64_t seq_off;      // index into the Seq arena
    uint32_t len, entry, last, adler;   // adler: the entry is a zlib stream (its Adler-32 partial sums are wanted)
    uint32_t nseq, nlit;
    uint32_t head_len, raw;        // raw: pieces = head + plain; else head + literals + tail (zstd) / body (deflate)
    uint32_t tail_off, tail_len;   // inside the body
    uint64_t litp_off;             // literal payload of a compressed zstd block: the literal arena (raw) or the body (Huffman)
    uint32_t litp_len, effort;     // effort: the entry's (enc_effort)
    uint64_t adler_a, adler_b;     // sum of bytes, sum of (len - k) * byte_k
};
// The `level` of the reference's writers (zstd 1..22, default 3: compress/zstandard.rs:46; deflate 0..9, default 6:
// compress/deflate.rs:89) selects one of this encoder's settings:
//   0 fast     greedy parse, Predefined FSE tables / fixed Huffman        zstd 1-2, deflate 1-3
//   1 default  greedy parse, per-block FSE tables / dynamic Huffman, chosen by cost   zstd 3-5 (and < 0 / 0 = default), deflate 4-6 (and < 0)
//   2 high     lazy parse (one position of look-ahead) + per-block FSE  zstd >= 6, deflate 7-9
//   3 stored   deflate level 0: stored blocks only
inline uint32_t enc_effort(uint8_t compression, int32_t level) {
    if (compression == 2) return level <= 0 ? 1u : level <= 2 ? 0u : level <= 5 ? 1u : 2u;
    if (compression == 1) return level < 0 ? 1u : level == 0 ? 3u : level <= 3 ? 0u : level <= 6 ? 1u : 2u;
    if (compression == 4) return level >= 0 && level <= 3 ? 1u : 2u;   // xz 0..9, default 6 (compress/xz.rs:10-16): presets >= 4 parse lazily, lc = 2 (0-3: lc = 0)
    return 1u;
}
constexpr uint32_t ENC_BLOCK_THREADS = 128;
constexpr uint32_t TMP_HEAD = 16;
// zstd: a new FRAME every FRAME_SEGS segments (1 MiB of input).  Blocks never reference earlier blocks here, so the split costs
// 6 bytes per MiB and nothing else; a reader that executes matches frame by frame (ours: one LZ unit per frame) gets
// parallelism inside long entries and solid streams, and zstd::Decoder reads concatenated frames (lib/src/entry/read.rs:181).
constexpr uint32_t FRAME_SEGS = 32;
constexpr uint32_t TMP_SEG = TMP_HEAD + SEG + SEG / 8 + 112;   // 36992: head + worst fixed-Huffman body, multiple of 16

struct EncEntry {
    uint64_t plain_off, plain_len;
    uint64_t piece_begin;          // first Segment of this entry's piece list
    uint64_t hdr_off;              // XZ_HDR_SCRATCH bytes in the work arena: frame header at +0, trailer at +16 (xz: +24)
    uint64_t out_off, out_cap;
    uint64_t comp_len, out_len;    // device written
    uint32_t seg_begin, n_segs;
    uint32_t n_pieces;             // device written
    int32_t key_idx;
    int32_t status;
    uint8_t compression, encryption, cipher_mode, effort;   // effort: enc_effort(compression, level)
    uint8_t iv[16];
    // GCM STREAM (cipher mode 2): segment size, this entry's ranges in the plan's segment / tile slot tables, stream header
    uint32_t gcm_seg_size, gcm_slot_begin, gcm_tile_begin, gcm_tiles_per_seg, gcm_pow_idx;
    uint8_t gcm_hdr[76];
};

constexpr int ENC_WARPS = 9;          // 9 warps x 8 KB of hash table per CTA, 3 CTAs per SM: 27 segments in flight per SM
constexpr int HLOG = 12;
// Only the hash table lives in shared memory.  The segment itself is read straight from HBM through L1/L2 (the step's own
// 32 positions are one coalesced row, candidates are sector reads that mostly hit L2): staging the 32 KiB segment in
// shared memory capped the kernel at 5 warps per SM, and the matcher is latency-bound -- warps in flight are what counts.
struct MatchSmem {
    uint16_t table[1 << HLOG];
};
constexpr uint32_t MATCH_SMEM_BYTES = (uint32_t)sizeof(MatchSmem) * ENC_WARPS;
static_assert(sizeof(MatchSmem) % 16 == 0, "16-byte aligned per warp");

__global__ void __launch_bounds__(32 * ENC_WARPS) lz_match_kernel(const uint8_t* __restrict__ work_ro, uint8_t* __restrict__ work,
                                                                  SegRec* __restrict__ segs, uint32_t nsegs, Seq* __restrict__ seqs) {
    extern __shared__ __align__(16) uint8_t match_smem_raw[];
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * ENC_WARPS + (threadIdx.x >> 5);
    if (s >= nsegs) return;
    MatchSmem* const S = reinterpret_cast<MatchSmem*>(match_smem_raw) + (threadIdx.x >> 5);
    const SegRec sr = segs[s];
    const uint32_t len = sr.len;
    // ---- clear the table; Adler partial sums over the segment (16-byte rows, coalesced)
    uint64_t ad_a = 0, ad_b = 0;
    {
        const uint4* src = reinterpret_cast<const uint4*>(work_ro + sr.plain_off);
        const uint32_t rows = (len + 15) / 16;
        for (uint32_t i = lane; i < (sr.adler ? rows : 0u); i += 32) {
            const uint4 v = __ldg(src + i);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t p0 = i * 16 + 4 * k;
                const uint32_t m = p0 + 4 <= len ? 0xFFFFFFFFu : p0 >= len ? 0u : (0xFFFFFFFFu >> (8 * (4 - (len - p0))));
                const uint32_t keep = w[k] & m;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const uint32_t byte = (keep >> (8 * b)) & 0xFF;
                    const uint32_t p = p0 + b;
                    ad_a += byte;
                    if (p < len) ad_b += (uint64_t)(len - p) * byte;
                }
            }
        }
        for (uint32_t i = lane; i < (1u << HLOG) * 2 / 16; i += 32) reinterpret_cast<uint4*>(S->table)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { ad_a += __shfl_xor_sync(0xFFFFFFFFu, ad_a, o); ad_b += __shfl_xor_sync(0xFFFFFFFFu, ad_b, o); }
    }
    __syncwarp();
    // the plain region is followed by the literal region of the same arena, so reads a few hundred bytes past the
    // segment stay inside the allocation; every length is clamped to the segment (maxlen)
    const uint8_t* const d = work_ro + sr.plain_off;   // 16-byte aligned
    auto ld32 = [&](uint32_t pos) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(d + (pos & ~3u));
        return __funnelshift_r(__ldg(q), __ldg(q + 1), (pos & 3u) * 8u);
    };
    Seq* const sq = seqs + sr.seq_off;
    uint8_t* const lits = work + sr.lit_off;
    uint32_t nseq = 0, nlit = 0, lit_at_last = 0;   // literals emitted before the last match
    uint32_t carry = 0;                              // first position of the next step that is not covered by a match
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t vn = ld32((uint32_t)lane);
    for (uint32_t base = 0; base < len; base += 32) {
        const uint32_t p = base + lane;
        const bool valid = p + 4 <= len;
        const uint32_t v = vn;                                 // the four bytes at p
        if (base + 32 < len) vn = ld32(p + 32);                // the next step's row, in flight during this step
        const uint32_t h = (v * 2654435761u) >> (32 - HLOG);
        const uint32_t ct = valid ? S->table[h] : 0xFFFFu;
        // one MATCH on the hash groups the lanes: the nearest lower lane of my group is the in-step candidate when its four
        // bytes really are mine (else a hash collision: no in-step candidate), the highest lane of each group inserts
        const uint32_t hm = __match_any_sync(0xFFFFFFFFu, valid ? h : (0x10000u | (unsigned)lane));
        const uint32_t lower = hm & lt;
        const int t1 = 31 - __clz((int)(lower | 1u));
        const uint32_t vt = __shfl_sync(0xFFFFFFFFu, v, t1);
        const uint32_t cw = (valid && lower && vt == v) ? base + (uint32_t)t1 : 0xFFFFu;
        __syncwarp();
        if (valid && lane == 31 - __clz((int)hm)) S->table[h] = (uint16_t)p;   // deterministic; every position is inserted
        if (carry >= 32) { carry -= 32; continue; }   // the whole step lies inside a match
        // ---- match lengths against both candidates in one loop (lengths are clamped to the segment, so the over-read
        // behind it is harmless)
        uint32_t best = 0, boff = 0;
        if (valid && (uint32_t)lane >= carry) {   // positions below `carry` lie inside the previous step's last match: never parsed
            const uint32_t maxlen = len - p < MAX_MATCH ? len - p : MAX_MATCH;
            bool aw = cw != 0xFFFFu, at = ct != 0xFFFFu && ct != cw;
            uint32_t lw = 0, ltb = 0, k = 0;
            // eight bytes per round (three aligned words + two funnel shifts per stream): candidate reads are L2 round
            // trips, so fewer, wider rounds
            auto ld64 = [&](uint32_t pos) -> uint64_t {
                const uint32_t* q = reinterpret_cast<const uint32_t*>(d + (pos & ~3u));
                const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2), sh = (pos & 3u) * 8u;
                return (uint64_t)__funnelshift_r(w0, w1, sh) | ((uint64_t)__funnelshift_r(w1, w2, sh) << 32);
            };
            while (k < maxlen && (aw || at)) {
                const uint64_t x = ld64(p + k);
                if (aw) { const uint64_t df = x ^ ld64(cw + k); if (df) { aw = false; lw = k + ((uint32_t)__ffsll((long long)df) - 1u) / 8u; } }
                if (at) { const uint64_t df = x ^ ld64(ct + k); if (df) { at = false; ltb = k + ((uint32_t)__ffsll((long long)df) - 1u) / 8u; } }
                k += 8;
            }
            if (aw) lw = maxlen;
            if (at) ltb = maxlen;
            lw = lw < maxlen ? lw : maxlen;
            ltb = ltb < maxlen ? ltb : maxlen;
            if (lw >= MIN_MATCH && lw >= ltb) { best = lw; boff = p - cw; }
            else if (ltb >= MIN_MATCH) { best = ltb; boff = p - ct; }
        }
        // lazy matching (high effort): a match gives way to a strictly longer one that starts at the next position -- its first
        // byte becomes a literal.  (Lane 31 cannot see its successor and stays greedy.)
        if (sr.effort >= 2u) {
            const uint32_t nb = __shfl_down_sync(0xFFFFFFFFu, best, 1);
            if (lane < 31 && best && nb > best) best = 0;
        }
        // ---- greedy parse of the step: orbit of `carry` under p -> p + (match ? len : 1), by pointer doubling
        uint32_t J = (uint32_t)lane + (best ? best : 1u);
        bool M = (uint32_t)lane >= carry;                      // no match anywhere in the step: everything from carry on is a literal
        if (__any_sync(0xFFFFFFFFu, best != 0)) {
            M = (uint32_t)lane == carry;
#pragma unroll
            for (int r = 0; r < 5; r++) {
                const uint32_t bits = (M && J < 32) ? (1u << J) : 0u;
                const uint32_t all = __reduce_or_sync(0xFFFFFFFFu, bits);
                M = M || ((all >> lane) & 1u);
                const uint32_t Jn = __shfl_sync(0xFFFFFFFFu, J, (int)(J & 31));
                J = J < 32 ? Jn : J;
            }
        } else J = 32;                                         // carry_out = 0
        const uint32_t carry_out = __shfl_sync(0xFFFFFFFFu, J, (int)carry) - 32u;
        const bool is_match = M && best != 0;
        const bool is_lit = M && best == 0 && p < len;
        const uint32_t mmask = __ballot_sync(0xFFFFFFFFu, is_match), lmask = __ballot_sync(0xFFFFFFFFu, is_lit);
        if (is_match) {
            const uint32_t prev = mmask & lt;
            uint32_t ll;
            if (prev) { const uint32_t pl = 31u - (uint32_t)__clz((int)prev); ll = (uint32_t)__popc(lmask & lt & ~((2u << pl) - 1u)); }
            else ll = (uint32_t)__popc(lmask & lt) + (nlit - lit_at_last);
            Seq q;
            q.off = boff;
            q.llml = ll | (best << 16);
            sq[nseq + (uint32_t)__popc(prev)] = q;
        }
        if (is_lit) lits[nlit + (uint32_t)__popc(lmask & lt)] = (uint8_t)v;
        if (mmask) {
            const uint32_t lastm = 31u - (uint32_t)__clz((int)mmask);
            lit_at_last = nlit + (uint32_t)__popc(lmask & ((1u << lastm) - 1u));
        }
        nseq += (uint32_t)__popc(mmask);
        nlit += (uint32_t)__popc(lmask);
        carry = carry_out;
    }
    if (lane == 0) {
        segs[s].nseq = nseq; segs[s].nlit = nlit;
        segs[s].adler_a = ad_a; segs[s].adler_b = ad_b;
    }
}

// ------------------------------------------------------------------------------------------------
// COMP: the codec this instantiation writes (2 zstd, 1 deflate); segments of the other codec are left to the other launch.  Two
// kernels because the deflate writer carries 6 KB of Huffman scratch and 80 registers: the zstd writer should not pay for them.
template <int COMP>
__global__ void __launch_bounds__(128) enc_block_kernel(uint8_t* __restrict__ work, SegRec* __restrict__ segs, uint32_t nsegs,
                                                        Seq* __restrict__ seqs, const EncTables* __restrict__ tables,
                                                        const EncEntry* __restrict__ entries) {
    __shared__ EncTables T;
    for (uint32_t i = threadIdx.x; i < sizeof(EncTables) / 4; i += blockDim.x)
        reinterpret_cast<uint32_t*>(&T)[i] = reinterpret_cast<const uint32_t*>(tables)[i];
    __syncthreads();
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsegs) return;
    SegRec& sr = segs[s];
    const uint32_t len = sr.len, nseq = sr.nseq, nlit = sr.nlit, last = sr.last;
    uint8_t* const head = work + sr.tmp_off;
    uint8_t* const body = head + TMP_HEAD;
    Seq* sq = seqs + sr.seq_off;
    if (entries[sr.entry].compression != COMP) return;
    if (COMP == 2) {
        // literals section first (Huffman-compressed into the body when that is smaller, else raw = the literal arena as it
        // is), the sequences section behind it on the next 4-byte boundary
        uint8_t lh[5];
        uint32_t lhn = 0;
        const uint32_t clit = zstd_write_literals(work + sr.lit_off, nlit, body, lh, &lhn);
        const uint32_t lpay = clit ? clit : nlit;
        const uint32_t sbase = clit ? (clit + 3u) & ~3u : 0u;
        uint32_t ssz = 1, soff = 0;
        bool fits = true;
        if (nseq) {
            zstd_assign_repcodes(sq, nseq);
            const uint32_t r = zstd_write_sequences(T, sq, nseq, body + sbase, TMP_SEG - TMP_HEAD - sbase, sr.effort >= 1u);
            if (r == 0xFFFFFFFFu) fits = false;
            soff = r >> 24; ssz = r & 0xFFFFFFu;
        } else body[sbase] = 0;
        const uint32_t csize = lhn + lpay + ssz;
        if (!fits || csize >= len) {
            zstd_block_header(last, 0, len, head);
            sr.head_len = 3; sr.raw = 1; sr.tail_off = 0; sr.tail_len = 0; sr.litp_off = 0; sr.litp_len = 0;
        } else {
            zstd_block_header(last, 2, csize, head);
            for (uint32_t k = 0; k < lhn; k++) head[3 + k] = lh[k];
            sr.head_len = 3 + lhn; sr.raw = 0; sr.tail_off = sbase + soff; sr.tail_len = ssz;
            sr.litp_off = clit ? sr.tmp_off + TMP_HEAD : sr.lit_off;
            sr.litp_len = lpay;
        }
    } else {
        // The writer's histogram / code tables (316 words) stay in the thread's local memory.  Shared memory was measured and is
        // slower here: 158 KB of tables per 128 threads leave one CTA per SM, and this lane-per-segment kernel lives on warps
        // in flight (block_write for 4 GiB: local 80 ms, shared rows 114 ms, fixed Huffman 21 ms).
        uint32_t ws_local[DEFLATE_WS];
        DeflateScratch scratch;
        const uint32_t sz = deflate_write_segment(sq, nseq, work + sr.lit_off, nlit, last != 0, body, sr.effort >= 1u && sr.effort != 3u, ws_local, 1, scratch);
        if (sz >= len + 5 || sr.effort == 3u) {   // effort 3: deflate level 0 = stored blocks
            head[0] = (uint8_t)(last ? 1 : 0); head[1] = (uint8_t)len; head[2] = (uint8_t)(len >> 8);
            head[3] = (uint8_t)~len; head[4] = (uint8_t)(~len >> 8);
            sr.head_len = 5; sr.raw = 1; sr.tail_off = 0; sr.tail_len = 0;
        } else { sr.head_len = 0; sr.raw = 0; sr.tail_off = 0; sr.tail_len = sz; }
    }
}

// ------------------------------------------------------------------------------------------------
// xz: a warp (= a CTA) per segment.  All lanes reset the segment's probability arena (16 KB of shared memory: the dependent
// load-update-store chain per coded bit runs at shared-memory latency) and take the CRC-32 of a 1 KiB slice each.  Then, sequence by
// sequence: the lanes turn 32 literals at a time into their coder events (lzma_enc_core.cuh: probability index and bit depend on
// data and parse only), lane 0 adds the events of the match, the warp resolves the events into probability VALUES (the adaptation
// of a slot depends on the order of the events on that slot only), and lane 0 runs the one serial loop that is left -- bound,
// low, range, normalise -- over the ring.
// Segments are independent chunks, so a 4 MiB file is 128 coders in flight; the arena decides how many per SM (lc = 2: 22, lc = 0: 43).
constexpr uint32_t XZ_ENC_RING = 32 * xz::EV_PER_LITERAL + xz::EV_PER_MATCH_MAX;   // 32 literals and the match behind them
__host__ __device__ constexpr uint32_t xz_lc_for_effort(uint32_t effort) { return effort <= 1u ? 0u : 2u; }
__host__ __device__ constexpr uint32_t xz_enc_smem_bytes(uint32_t lc) { return ((xz::enc_probs(lc) + 2 + XZ_ENC_RING) * 2u + 15u) & ~15u; }
// one launch per literal-context setting (lc): the arena size is a launch parameter
__global__ void __launch_bounds__(32) xz_encode_kernel(uint8_t* __restrict__ work, SegRec* __restrict__ segs, uint32_t nsegs,
                                                       const Seq* __restrict__ seqs, const EncEntry* __restrict__ entries, uint32_t lc) {
    extern __shared__ __align__(16) uint8_t xz_enc_smem_raw[];
    const uint32_t lane = threadIdx.x;
    const uint32_t s = blockIdx.x;
    if (s >= nsegs) return;
    SegRec& sr = segs[s];
    if (entries[sr.entry].compression != 4 || xz_lc_for_effort(sr.effort) != lc) return;
    const uint32_t n_probs = xz::enc_probs(lc);
    uint16_t* const probs = reinterpret_cast<uint16_t*>(xz_enc_smem_raw);
    uint16_t* const ring = probs + n_probs + 2;
    for (uint32_t i = lane; i < n_probs; i += 32) probs[i] = (uint16_t)xz::PROB_INIT;
    const uint32_t len = sr.len;
    const uint8_t* const d = work + sr.plain_off;
    const uint32_t lo = lane * (SEG / 32), nl = lo >= len ? 0u : (len - lo < SEG / 32 ? len - lo : SEG / 32);
    const uint32_t my_crc = nl ? xz::crc_slice(d + lo, nl) : 0u;
    const uint32_t my_pow = xz::crc_xpow_bytes(nl);
    uint32_t crc = 0;
    for (int l = 0; l < 32; l++) {
        const uint32_t c = __shfl_sync(0xFFFFFFFFu, my_crc, l), pw = __shfl_sync(0xFFFFFFFFu, my_pow, l);
        crc = xz::crc_concat(crc, c, pw);
    }
    __syncwarp();
    uint8_t* const head = work + sr.tmp_off;
    const uint32_t cap = len > 4 ? len - 4 : 0u;   // a compressed chunk must save its three extra header bytes
    xz::RangeEnc rc;                               // lane 0's copy is the coder
    rc.init(head + TMP_HEAD, head + TMP_HEAD + cap, head + TMP_SEG);
    uint32_t state = 0, rep0 = 0, rep1 = 0, rep2 = 0, rep3 = 0, pos = 0;   // the same in every lane
    const Seq* const sq = seqs + sr.seq_off;
    const uint32_t nseq = cap ? sr.nseq : 0u;
    bool over = cap == 0;
    // one round per sequence, and a last one for the literals behind the last match; ONE call site of the coder loop
    for (uint32_t q = 0; q <= nseq && !over; q++) {
        const bool has_match = q < nseq;
        uint32_t ll = len - pos, ml = 0, dist = 0;
        if (has_match) { const Seq v = sq[q]; ll = v.llml & 0xFFFFu; ml = v.llml >> 16; dist = v.off - 1u; }
        const uint32_t rep0_lit = rep0;   // the first literal behind a match looks at the byte at the LAST distance
        const uint32_t kind = has_match ? xz::rep_classify(dist, rep0, rep1, rep2, rep3) : 0u;
        uint32_t base = 0;
        do {
            const uint32_t j = base + lane, p = pos + j, cnt = ll - base < 32 ? ll - base : 32;
            if (j < ll) {
                const uint32_t st = xz::lit_state_after(state, j);
                xz::gen_literal_events(ring + lane * xz::EV_PER_LITERAL, p, d[p], p ? d[p - 1] : 0u, st, st >= 7 ? d[p - rep0_lit - 1] : 0u, lc);
            }
            uint32_t total = cnt * xz::EV_PER_LITERAL;
            if (lane == 0 && has_match && base + 32 >= ll)
                total += xz::gen_match_events(ring + total, pos + ll, xz::lit_state_after(state, ll), kind, ml, dist);
            total = __shfl_sync(0xFFFFFFFFu, total, 0);
            __syncwarp();
            // events -> values: 32 events per round trip; lanes whose events hit the same probability slot take turns in event order
            for (uint32_t b0 = 0; b0 < total; b0 += 32) {
                const uint32_t i = b0 + lane;
                const bool live = i < total;
                const uint32_t ev = live ? ring[i] : 0u, bit = ev >> 15, idx = ev & xz::EV_INDEX;
                const bool coded = live && !(ev & xz::EV_DIRECT);
                const uint32_t grp = __match_any_sync(0xFFFFFFFFu, coded ? idx : (0x10000u | lane));
                const uint32_t rank = (uint32_t)__popc(grp & ((1u << lane) - 1u));
                const uint32_t rounds = __reduce_max_sync(0xFFFFFFFFu, coded ? (uint32_t)__popc(grp) : 1u);
                uint32_t v = 0;
                for (uint32_t r = 0; r < rounds; r++) {
                    if (coded && rank == r) { v = probs[idx]; probs[idx] = (uint16_t)xz::prob_step(v, bit); }
                    __syncwarp();
                }
                if (live) ring[i] = (uint16_t)(coded ? (v | (bit << 15)) : (xz::EV_DIRECT | (bit << 15)));
            }
            __syncwarp();
            if (lane == 0) xz::code_values(rc, ring, total);
            __syncwarp();
            base += 32;
        } while (base < ll);
        state = xz::lit_state_after(state, ll);
        if (has_match) state = xz::match_state_next(state, kind);
        pos += ll + ml;
        over = __shfl_sync(0xFFFFFFFFu, rc.over ? 1 : 0, 0) != 0;
    }
    if (lane) return;
    rc.flush();
    const uint32_t cs = (over || rc.over || (uint32_t)(rc.p - (head + TMP_HEAD)) > cap) ? 0xFFFFFFFFu : (uint32_t)(rc.p - (head + TMP_HEAD));
    if (cs == 0xFFFFFFFFu) { sr.head_len = xz::lzma2_chunk_header(head, len, 0, lc); sr.raw = 1; sr.tail_off = 0; sr.tail_len = 0; }
    else { sr.head_len = xz::lzma2_chunk_header(head, len, cs, lc); sr.raw = 0; sr.tail_off = 0; sr.tail_len = cs; }
    sr.adler_a = crc;
}

// ------------------------------------------------------------------------------------------------
__global__ void enc_layout_kernel(uint8_t* __restrict__ work, const SegRec* __restrict__ segs, EncEntry* __restrict__ entries,
                                  uint32_t n, Segment* __restrict__ pieces) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    EncEntry& e = entries[i];
    if (e.status != ST_OK) { e.comp_len = 0; e.n_pieces = 0; return; }
    Segment* P = pieces + e.piece_begin;
    uint64_t pos = 0;
    uint32_t np = 0;
    auto add = [&](uint64_t off, uint64_t len) { if (len) { P[np].img_off = off; P[np].pos = pos; np++; pos += len; } };
    uint8_t* h = work + e.hdr_off;
    if (e.compression == 0) add(e.plain_off, e.plain_len);
    else if (e.compression == 2) {
        h[0] = 0x28; h[1] = 0xB5; h[2] = 0x2F; h[3] = 0xFD; h[4] = 0x00; h[5] = 0x38;
        if (e.n_segs == 0) { zstd_block_header(1, 0, 0, h + 6); add(e.hdr_off, 9); }
        for (uint32_t k = e.seg_begin; k < e.seg_begin + e.n_segs; k++) {
            const SegRec& s = segs[k];
            if ((k - e.seg_begin) % FRAME_SEGS == 0) add(e.hdr_off, 6);   // frame header (the same six bytes every time)
            add(s.tmp_off, s.head_len);
            if (s.raw) add(s.plain_off, s.len);
            else { add(s.litp_off, s.litp_len); add(s.tmp_off + TMP_HEAD + s.tail_off, s.tail_len); }
        }
    } else if (e.compression == 4) {
        // .xz container around the segments' LZMA2 chunks (lzma_enc_core.cuh): front at +0, back at +24 of the entry's scratch
        const bool empty = e.n_segs == 0;
        add(e.hdr_off, xz::xz_write_front(h, empty));
        uint64_t chunk_bytes = 0;
        uint32_t crc = 0;
        const uint32_t pow_seg = xz::crc_xpow_bytes(SEG);
        for (uint32_t k = e.seg_begin; k < e.seg_begin + e.n_segs; k++) {
            const SegRec& s = segs[k];
            add(s.tmp_off, s.head_len);
            if (s.raw) add(s.plain_off, s.len); else add(s.tmp_off + TMP_HEAD, s.tail_len);
            chunk_bytes += s.head_len + (s.raw ? s.len : s.tail_len);
            crc = xz::crc_concat(crc, (uint32_t)s.adler_a, s.len == SEG ? pow_seg : xz::crc_xpow_bytes(s.len));
        }
        add(e.hdr_off + 24, xz::xz_write_back(h + 24, empty, chunk_bytes, e.plain_len, crc));
    } else {
        h[0] = 0x78; h[1] = 0x9C;
        if (e.n_segs == 0) { h[2] = 0x03; h[3] = 0x00; add(e.hdr_off, 4); }
        else add(e.hdr_off, 2);
        uint64_t a = 1, b = e.plain_len % 65521u, o = 0;
        for (uint32_t k = e.seg_begin; k < e.seg_begin + e.n_segs; k++) {
            const SegRec& s = segs[k];
            if (s.raw) { add(s.tmp_off, s.head_len); add(s.plain_off, s.len); }
            else add(s.tmp_off + TMP_HEAD, s.tail_len);
            a = (a + s.adler_a) % 65521u;
            const uint64_t rest = (e.plain_len - o - s.len) % 65521u;
            b = (b + s.adler_b % 65521u + rest * (s.adler_a % 65521u)) % 65521u;
            o += s.len;
        }
        const uint32_t ad = (uint32_t)((b << 16) | a);
        h[16] = (uint8_t)(ad >> 24); h[17] = (uint8_t)(ad >> 16); h[18] = (uint8_t)(ad >> 8); h[19] = (uint8_t)ad;
        add(e.hdr_off + 16, 4);
    }
    e.n_pieces = np;
    e.comp_len = pos;
    const uint64_t hdr = e.encryption ? 16 : 0;
    if (e.encryption && e.cipher_mode == 2) {   // header || { segment || tag }: full segments while data follows, then a final one (gcm.rs:44-90)
        const uint64_t S = e.gcm_seg_size, nseg = pos ? (pos + S - 1) / S : 1;
        e.out_len = gcm::GCM_HEADER_LEN + pos + nseg * gcm::GCM_TAG_LEN;
    } else
    e.out_len = e.encryption && e.cipher_mode == 0 ? hdr + (pos / 16 + 1) * 16 : hdr + pos;
    if (e.out_len > e.out_cap) { e.status = ST_NOSPACE; }
}

// ------------------------------------------------------------------------------------------------
// CTR encrypt (or plain gather) of the piece list into the output: out = [IV |] E_K(IV + i) ^ stream.
// Tiles are built on the host from the stream-length BOUND; blocks past the produced length do nothing.
template <int ENC /*0 none, 1 aes, 2 camellia*/>
__global__ void __launch_bounds__(ENC == 1 ? AES_CTR_THREADS : 256) encrypt_tiles_kernel(const uint8_t* __restrict__ work, const Segment* __restrict__ pieces,
                                                            const EncEntry* __restrict__ entries,
                                                            const CipherTile* __restrict__ tiles, uint32_t n_tiles,
                                                            const DevKeys* __restrict__ keys, const AesTables* __restrict__ aes,
                                                            const CamelliaTables* __restrict__ cam, uint8_t* __restrict__ out) {
    extern __shared__ uint32_t smem[];
    uint32_t* s_tab = smem;
    if (ENC == 1) aes_te4_fill(s_tab, aes);   // four lane-replicated tables, 1024 threads per CTA (see aes_ctr_tiles_kernel)
    else if (ENC == 2) {
        for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_tab[i] = (&cam->sp_hi[0][0])[i]; s_tab[2048 + i] = (&cam->sp_lo[0][0])[i]; }
    }
    __shared__ uint32_t s_key32[60];
    __shared__ uint64_t s_key64[34];
    __shared__ int s_key_idx;
    if (threadIdx.x == 0) s_key_idx = -2;
    __syncthreads();
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const CipherTile tl = tiles[t];
        const EncEntry& e = entries[tl.entry];
        if (e.status != ST_OK) continue;
        const uint64_t clen = e.comp_len;
        if (ENC != 0 && e.key_idx != s_key_idx) {
            __syncthreads();
            const DevKeys* k = keys + e.key_idx;
            if (ENC == 1) { if (threadIdx.x < 60) s_key32[threadIdx.x] = k->aes_rk[threadIdx.x]; }
            else { if (threadIdx.x < 34) s_key64[threadIdx.x] = k->cam_ek[threadIdx.x]; }
            if (threadIdx.x == 0) s_key_idx = e.key_idx;
            __syncthreads();
        }
        const Segment* sg = pieces + e.piece_begin;
        uint8_t* dst = out + e.out_off + (ENC ? 16 : 0);
        uint32_t iv[4] = {0, 0, 0, 0};
        if (ENC) {
            for (int k = 0; k < 16; k++) iv[k >> 2] |= (uint32_t)e.iv[k] << (8 * (k & 3));
            if (tl.first_block == 0 && threadIdx.x < 16) out[e.out_off + threadIdx.x] = e.iv[threadIdx.x];
        }
        for (uint32_t j = threadIdx.x; j < tl.n_blocks; j += blockDim.x) {
            const uint64_t bi = tl.first_block + j;
            if (bi * 16 >= clen) break;
            const uint32_t have = (uint32_t)(clen - bi * 16 >= 16 ? 16 : clen - bi * 16);
            uint32_t c[4] = {0, 0, 0, 0};
            if (have == 16) load_stream16(work, sg, e.n_pieces, clen, bi * 16, c);
            else for (uint32_t k = 0; k < have; k++) c[k >> 2] |= (uint32_t)load_stream1(work, sg, e.n_pieces, bi * 16 + k) << (8 * (k & 3));
            uint32_t o[4] = {c[0], c[1], c[2], c[3]};
            if (ENC != 0) {
                ctr128be_add(iv, bi, o);
                if (ENC == 1) aes256_encrypt_block4(o, s_key32, LaneTe4{reinterpret_cast<const uint8_t*>(s_tab), (threadIdx.x & 31) * 4});
                else camellia256_crypt_block(o, s_key64, s_tab, s_tab + 2048);
                o[0] ^= c[0]; o[1] ^= c[1]; o[2] ^= c[2]; o[3] ^= c[3];
            }
            if (have == 16) *reinterpret_cast<uint4*>(dst + bi * 16) = make_uint4(o[0], o[1], o[2], o[3]);
            else for (uint32_t k = 0; k < have; k++) dst[bi * 16 + k] = (uint8_t)(o[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// CBC encrypt: C_i = E_K(P_i ^ C_{i-1}), PKCS#7 always appends (lib/src/cipher/block/write.rs:48-57,124).
// One lane per entry -- the chain is serial; list[] = indices of the CBC entries of this cipher.
template <int ENC>
__global__ void __launch_bounds__(64) cbc_encrypt_kernel(const uint8_t* __restrict__ work, const Segment* __restrict__ pieces,
                                                         const EncEntry* __restrict__ entries, const uint32_t* __restrict__ list,
                                                         uint32_t n, const DevKeys* __restrict__ keys,
                                                         const AesTables* __restrict__ aes, const CamelliaTables* __restrict__ cam,
                                                         uint8_t* __restrict__ out) {
    extern __shared__ uint32_t smem[];
    uint32_t* s_tab = smem;
    if (ENC == 1) { for (int i = threadIdx.x; i < 256 * 32; i += blockDim.x) s_tab[i] = aes->te0[i >> 5]; }
    else { for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_tab[i] = (&cam->sp_hi[0][0])[i]; s_tab[2048 + i] = (&cam->sp_lo[0][0])[i]; } }
    __syncthreads();
    const TabView tv{s_tab, 32, (uint32_t)(threadIdx.x & 31)};
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const EncEntry& e = entries[list[i]];
    if (e.status != ST_OK) return;
    const DevKeys* k = keys + e.key_idx;
    const Segment* sg = pieces + e.piece_begin;
    const uint64_t clen = e.comp_len, nblk = clen / 16 + 1;
    uint8_t* dst = out + e.out_off;
    uint32_t prev[4] = {0, 0, 0, 0};
    for (int q = 0; q < 16; q++) { prev[q >> 2] |= (uint32_t)e.iv[q] << (8 * (q & 3)); dst[q] = e.iv[q]; }
    for (uint64_t bi = 0; bi < nblk; bi++) {
        uint32_t c[4] = {0, 0, 0, 0};
        if ((bi + 1) * 16 <= clen) load_stream16(work, sg, e.n_pieces, clen, bi * 16, c);
        else {
            const uint32_t have = (uint32_t)(clen - bi * 16), pad = 16 - have;
            for (uint32_t q = 0; q < 16; q++) {
                const uint32_t b = q < have ? load_stream1(work, sg, e.n_pieces, bi * 16 + q) : pad;
                c[q >> 2] |= b << (8 * (q & 3));
            }
        }
        c[0] ^= prev[0]; c[1] ^= prev[1]; c[2] ^= prev[2]; c[3] ^= prev[3];
        if (ENC == 1) aes256_encrypt_block(c, k->aes_rk, tv);
        else camellia256_crypt_block(c, k->cam_ek, s_tab, s_tab + 2048);
        *reinterpret_cast<uint4*>(dst + 16 + bi * 16) = make_uint4(c[0], c[1], c[2], c[3]);
        prev[0] = c[0]; prev[1] = c[1]; prev[2] = c[2]; prev[3] = c[3];
    }
}

// FDAT-body CRC tiles come from the host with bound-based geometry: tile = bytes [rel, rel + cap) of entry
// tl.span's output (span field reused as entry index until clipped).  Clip to the produced length.
struct CrcTileSrc { uint64_t rel; uint32_t cap, entry, span; };
__global__ void crc_clip_kernel(const CrcTileSrc* __restrict__ src, uint32_t n, const EncEntry* __restrict__ entries,
                                CrcTile* __restrict__ tiles) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const CrcTileSrc s = src[i];
    const EncEntry& e = entries[s.entry];
    const uint64_t end = e.status == ST_OK ? e.out_len : 0;
    uint64_t len = s.rel < end ? end - s.rel : 0;
    if (len > s.cap) len = s.cap;
    CrcTile t;
    t.begin = len ? e.out_off + s.rel : e.out_off;   // empty tiles stay inside the arena (16-byte aligned: no load at all)
    t.len = (uint32_t)len;
    t.span = s.span;
    tiles[i] = t;
}

// GCM: the segment / tile tables are sized from the compressed-length BOUND on the host; once the produced length is known
// every slot is filled in (or marked unused) here, and slot 0 of an entry puts the stream header in front of its output.
struct GcmSlot { uint32_t entry, j; };
__global__ void gcm_enc_slots_kernel(const GcmSlot* __restrict__ slots, uint32_t n, const EncEntry* __restrict__ entries,
                                     gcm::GcmSeg* __restrict__ gsegs, gcm::GcmTile* __restrict__ tiles, uint8_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const GcmSlot sl = slots[i];
    const EncEntry& e = entries[sl.entry];
    const uint64_t S = e.gcm_seg_size;
    const uint32_t tps = e.gcm_tiles_per_seg, t0 = e.gcm_tile_begin + sl.j * tps;
    const uint64_t nseg = e.status != ST_OK ? 0 : e.comp_len ? (e.comp_len + S - 1) / S : 1;
    gcm::GcmSeg g;
    memset(&g, 0, sizeof g);
    uint32_t used = 0;
    if (sl.j >= nseg) g.ct_len = gcm::GCM_SEG_UNUSED;
    else {
        g.entry = sl.entry; g.pow_idx = e.gcm_pow_idx; g.key_idx = e.key_idx; g.enc = e.encryption;
        uint8_t nonce[12];
        for (int k = 0; k < 7; k++) nonce[k] = e.gcm_hdr[32 + k];
        nonce[7] = (uint8_t)(sl.j >> 24); nonce[8] = (uint8_t)(sl.j >> 16); nonce[9] = (uint8_t)(sl.j >> 8); nonce[10] = (uint8_t)sl.j;
        nonce[11] = sl.j + 1 == nseg ? 1 : 0;   // aead.rs:210-217
        for (int k = 0; k < 3; k++) g.nonce[k] = load_le32(nonce + 4 * k);
        g.src_seg_begin = e.piece_begin; g.src_n_segs = e.n_pieces; g.src_len = e.comp_len;
        g.ct_pos = (uint64_t)sl.j * S;
        g.ct_len = e.comp_len - g.ct_pos < S ? e.comp_len - g.ct_pos : S;
        g.dst_off = e.out_off + gcm::GCM_HEADER_LEN + (uint64_t)sl.j * (S + gcm::GCM_TAG_LEN);
        g.first_tile = t0;
        const uint64_t nb = (g.ct_len + 15) / 16, head = nb % gcm::GCM_TILE_BLOCKS;
        uint64_t b0 = 0;
        if (head) { tiles[t0 + used++] = gcm::GcmTile{i, (uint32_t)head, 0}; b0 = head; }
        for (; b0 < nb; b0 += gcm::GCM_TILE_BLOCKS) tiles[t0 + used++] = gcm::GcmTile{i, gcm::GCM_TILE_BLOCKS, b0};
        g.n_tiles = used;
        if (sl.j == 0) for (uint32_t k = 0; k < gcm::GCM_HEADER_LEN; k++) out[e.out_off + k] = e.gcm_hdr[k];
    }
    for (uint32_t t = used; t < tps; t++) tiles[t0 + t] = gcm::GcmTile{i, 0, 0};
    gsegs[i] = g;
}

// host-side plan state (encode_host.cuh)
struct EncodePlan;
void destroy(EncodePlan* p);
bool init_attributes();

}  // namespace enc
}  // namespace pna
