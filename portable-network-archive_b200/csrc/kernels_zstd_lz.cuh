// kernels_zstd_lz.cuh -- LZ execution stage of the zstd decoder (K4): ONE CTA of W warps per entry.
//
// A frame's blocks are order-dependent through the window, so the parallelism inside an entry is the bytes
// and sequences of one STEP: 32*W consecutive sequences (<= STEP output bytes) handled by 32*W threads.
//   phase A  setup(s):    every thread writes, for each output byte of its sequence, a SOURCE CODE into idx[]:
//                         a step-relative position (a byte this same step produces) or FLAG | shared-memory offset of
//                         a byte that exists already (staged literal, older window byte).  Matches whose source has
//                         left the window ("far", offset > KEEP) were fetched from HBM one step ahead into registers
//                         and are stored straight into the window; overlapping matches (offset < length) get
//                         periodic codes, so chains never run inside one match.
//            front1(s+1): the next step's sequences from the cp.async-staged ring, per-warp packed scan of
//                         (literal length, total length), published to shared memory.
//   ---- barrier
//   phase B  resolve(s):  byte-parallel and divergence-free -- every thread chases idx[] down to an existing byte
//                         and copies it into the window (codes strictly decrease along a chain).
//            front2(s+1): cross-warp bases, the cut (first long sequence / STEP overflow), positions, offset
//                         validation, HBM fetch of far sources for the next step.
//   ---- barrier (also OR-reduces the offset-validation flags)
// The window is linear: when it fills, the newest KEEP bytes slide to the front (through registers).  Finished
// 512-byte rows stream to HBM as 16-byte stores, rows distributed over the warps.  Sequences longer than SEQ_MAX
// (or far matches > FAR_MAX bytes) go one at a time through whole-CTA copies.
//
// Two instantiations: LzSmall (4 warps, 16-bit codes, 29 KB of shared memory: 7 CTAs = 28 warps per SM, one wave
// for 1024 entries on 148 SMs) and LzBig (16 warps, 32-bit codes, 128 KiB window) for batches with fewer entries
// than SMs -- a solid archive is ONE frame.
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"
#include "zstd_core.cuh"
#include "kernels_crc_cipher.cuh"   // load16_any

namespace pna {
namespace zs {

struct ZEntry {          // per zstd entry, device resident
    uint32_t entry;      // index into EntryRec[]
    uint32_t blk_begin;  // first ZBlock
    uint32_t blk_count;
    uint32_t n_frames;   // device-written by zstd_resolve: frames that own at least one block
    uint64_t lit_base;   // literal arena base of this entry
    uint64_t seq_base;   // sequence array base
    uint64_t lit_total;  // device-written by zstd_resolve
    uint64_t seq_total;
    uint32_t unit_begin; // first LzUnit of this entry (host prefix sum of n_frames)
    uint32_t _pad;
};
// One unit of the LZ stage = one FRAME: matches never reach across a frame start, so the frames of a stream that is a
// concatenation of frames (what this library's own writer emits for long entries, and any multi-frame zstd stream) are
// executed by different CTAs.  A reference-written entry is one frame = one unit.
struct LzUnit { uint32_t ze, blk_begin, blk_count, _pad; };

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}
constexpr uint32_t LZ_SEQ_MAX = 255;   // ll and ml bound of the parallel path
constexpr uint32_t LZ_FAR_MAX = 32;    // far matches up to this length are prefetched (9 words)

template <int W_, typename Code_, uint32_t BUF_, uint32_t KEEP_, uint32_t STEP_, uint32_t LIT_RING_, uint32_t LIT_CH_, int CTAS_>
struct LzCfg {
    using Code = Code_;
    static constexpr int W = W_, CTAS = CTAS_;
    static constexpr uint32_t T = 32u * W_;
    static constexpr Code FLAG = (Code)((Code)1 << (8 * sizeof(Code) - 1));
    static constexpr uint32_t BUF = BUF_, KEEP = KEEP_, STEP = STEP_;
    static constexpr uint32_t SEQ_RING = 4 * T;                                  // four chunks of T sequences
    static constexpr uint32_t LIT_CH = LIT_CH_;                                  // literal bytes staged per pass (<= 16 * T)
    static constexpr uint32_t LIT_RING = LIT_RING_, LIT_GUARD = 256;
    static constexpr uint32_t OFF_IDX = BUF;
    static constexpr uint32_t OFF_SEQ = OFF_IDX + (STEP + 8) * (uint32_t)sizeof(Code);   // idx[] is indexed from the aligned window word of the step start
    static constexpr uint32_t OFF_LIT = OFF_SEQ + SEQ_RING * 8;
    static constexpr uint32_t OFF_SCAN = OFF_LIT + LIT_RING + LIT_GUARD;
    static constexpr uint32_t OFF_MISC = OFF_SCAN + (uint32_t)W * 32 * 4;
    static constexpr uint32_t BYTES = OFF_MISC + 64 + (uint32_t)W * 4;
    static_assert((LIT_RING & (LIT_RING - 1)) == 0 && LIT_RING >= STEP + LIT_CH, "literal ring covers one step plus one staged chunk");
    static_assert(KEEP >= 2 * STEP + 544, "far sources fetched one step ahead are already in HBM");
    static_assert(BUF >= KEEP + STEP + 32 && BUF >= KEEP + T + 32, "room for a step after a slide");
    static_assert(OFF_LIT + LIT_RING + LIT_GUARD < (uint64_t)FLAG, "codes address the CTA's shared block");
    static_assert(BUF - STEP - KEEP >= 16 * T && T <= STEP, "a slide moves the window by at least one round of pieces");
    static_assert(LIT_CH <= 16 * T && (LIT_CH & (LIT_CH - 1)) == 0, "one 16-byte piece per thread and pass");
};
using LzSmall = LzCfg<4, uint16_t, 16384, 8192, 3072, 4096, 1024, 7>;
using LzBig = LzCfg<16, uint32_t, 131072, 65536, 8192, 16384, 4096, 1>;

// n consecutive codes code, code+1, ... at ix: two (16-bit) codes per 32-bit store once ix is word aligned
template <typename Code>
__device__ __forceinline__ void fill_codes(Code* ix, uint32_t n, uint32_t code) {
    if constexpr (sizeof(Code) == 2) {
        if (n && (reinterpret_cast<uintptr_t>(ix) & 2)) { *ix++ = (Code)code; code++; n--; }
        uint32_t pair = code | ((code + 1) << 16);         // no carry between the halves: codes stay below 2^16
        uint32_t* p32 = reinterpret_cast<uint32_t*>(ix);
        for (uint32_t q = 0; q + 2 <= n; q += 2) { *p32++ = pair; pair += 0x00020002u; }   // (four codes per 64-bit store measured slower: 17.4 -> 18.0 ms)
        if (n & 1) ix[n - 1] = (Code)(code + n - 1);
    } else {   // 32-bit codes: two per 64-bit store once ix is 8-byte aligned
        if (n && (reinterpret_cast<uintptr_t>(ix) & 4)) { *ix++ = (Code)code; code++; n--; }
        uint2* p64 = reinterpret_cast<uint2*>(ix);
        for (uint32_t q = 0; q + 2 <= n; q += 2) { *p64++ = make_uint2(code + q, code + q + 1); }
        if (n & 1) ix[n - 1] = (Code)(code + n - 1);
    }
}

template <class C>
__global__ void __launch_bounds__(C::T, C::CTAS) zstd_lz_kernel(const uint8_t* __restrict__ buf, EntryRec* entries,
                                                               const ZEntry* __restrict__ ze, const uint32_t* __restrict__ order,
                                                               const LzUnit* __restrict__ units /* null: one unit per ZEntry */,
                                                               uint32_t nz, const ZBlock* __restrict__ blocks,
                                                               const uint8_t* __restrict__ lits, const SeqRec* __restrict__ seqs,
                                                               uint8_t* out) {
    using Code = typename C::Code;
    constexpr uint32_t T = C::T;
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    extern __shared__ __align__(16) uint8_t lz_smem[];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint8_t* const win = lz_smem;
    Code* const idx = reinterpret_cast<Code*>(lz_smem + C::OFF_IDX);
    SeqRec* const sring = reinterpret_cast<SeqRec*>(lz_smem + C::OFF_SEQ);
    uint8_t* const lring = lz_smem + C::OFF_LIT;
    uint32_t* const scan = reinterpret_cast<uint32_t*>(lz_smem + C::OFF_SCAN);   // [W][32] packed (lit << 16 | total) inclusive
    uint32_t* const misc = reinterpret_cast<uint32_t*>(lz_smem + C::OFF_MISC);   // [0..2] broadcast slot, [16..16+W) warp stops
    uint32_t* const wstop = misc + 16;

    if (blockIdx.x >= nz) return;
    const uint32_t ui = order ? order[blockIdx.x] : blockIdx.x;
    uint32_t zi = ui, blk_first = 0, blk_end = 0;
    if (units) { const LzUnit unit = units[ui]; zi = unit.ze; blk_first = unit.blk_begin; blk_end = unit.blk_begin + unit.blk_count; }
    const ZEntry* const zp = ze + zi;
    if (!units) { blk_first = zp->blk_begin; blk_end = blk_first + zp->blk_count; }
    EntryRec& er = entries[zp->entry];
    if (er.status != ST_OK) return;
    if (er.out_len > er.out_cap) { if (tid == 0) atomicCAS(&er.status, ST_OK, ST_NOSPACE); return; }
    // Positions are 32-bit and relative to the start of the CURRENT block (oblk = its place in HBM); they are rebased
    // at every block, so the window start and the flush mark may be negative.  oblk + bpos and oblk + flushed stay
    // multiples of 16 in the (16-byte aligned) entry.
    // A unit that is not the first frame of its entry starts at any byte: the window then begins `skip` bytes before it (at
    // the 16-byte boundary below), and those bytes -- another CTA's -- must never be written.  The regular flushes start
    // behind that first 16-byte group; its own bytes go out once, bytewise, from warp 0 in the first flush after the group is
    // complete (far matches read HBM, so it cannot wait long) or at the end of a unit shorter than that.
    // The pending mark lives in shared memory (misc[3]): the kernel has no register to spare.
    const uint64_t unit_off = (units && blk_end > blk_first) ? blocks[blk_first].out_off : 0;
    const uint32_t skip0 = (uint32_t)(unit_off & 15u);
    uint8_t* oblk = out + er.out_off + (unit_off - skip0);
    int32_t bpos = 0;                         // position of win[0]
    int32_t cur = (int32_t)skip0;             // position of the next output byte
    int32_t flushed = skip0 ? 16 : 0;         // HBM holds everything below (bar the pending head group)
    if (tid == 0) misc[3] = skip0;
    __syncthreads();
    // win[0] <-> oblk + bpos as long as the window has not slid
    auto flush_head = [&](bool at_end) {
        if (warp == 0) {
            const uint32_t a = misc[3];
            __syncwarp();
            const uint32_t have = (uint32_t)(cur - bpos);
            if (a && (at_end || have >= 16u)) {
                const uint32_t top = have < 16u ? have : 16u;
                if (lane >= a && lane < top) (oblk + (int64_t)bpos)[lane] = win[lane];
                if (lane == 0) misc[3] = 0;
            }
            __syncwarp();   // a second call in the same flush must see the cleared mark
        }
    };

    // ---- whole-CTA helpers; every one is called under uniform control flow
    // finished 512-byte rows -> HBM (rows distributed over the warps).  force: also the 16-byte groups and the byte
    // tail below cur (rewritten later with the same values).  Callers guarantee the window bytes are visible.
    auto flush = [&](bool force) {
        if (force) flush_head(true);
        if (flushed + 512 <= cur) {
            const uint32_t nrows = (uint32_t)((cur - flushed) >> 9);
            const uint32_t w0 = (uint32_t)(flushed - bpos);
            if (w0 == 16u) flush_head(false);   // the first row flush of a unit with a pending head group starts here (others: no-op)
            uint8_t* const g = oblk + (int64_t)flushed;
            for (uint32_t r = warp; r < nrows; r += C::W) {
                const uint4 v = *reinterpret_cast<const uint4*>(win + w0 + (r << 9) + 16 * lane);
                *reinterpret_cast<uint4*>(g + (r << 9) + 16 * lane) = v;
            }
            flushed += (int32_t)(nrows << 9);
        }
        if (force && flushed < cur) {
            const uint32_t n = (uint32_t)(cur - flushed);   // < 512
            const uint32_t w0 = (uint32_t)(flushed - bpos);
            if (warp == 0) {
                uint8_t* const g = oblk + (int64_t)flushed;
                if (16u * lane + 16u <= n) {
                    const uint4 v = *reinterpret_cast<const uint4*>(win + w0 + 16 * lane);
                    *reinterpret_cast<uint4*>(g + 16 * lane) = v;
                }
                const uint32_t full = n & ~15u;
                if (full + lane < n) g[full + lane] = win[w0 + full + lane];
            }
            flushed += (int32_t)(n & ~15u);
        }
    };
    // make room for `need` more bytes: the newest KEEP bytes (16-byte granular) slide to the front, through registers
    auto reserve = [&](uint32_t need) {
        if ((uint32_t)(cur - bpos) + need <= C::BUF) return;
        __syncthreads();
        flush(false);
        __syncthreads();
        const uint32_t fill = (uint32_t)(cur - bpos);
        const uint32_t shift = (fill - C::KEEP) & ~15u;       // fill > BUF - need >= KEEP + 32
        const uint32_t n16 = (fill - shift + 15u) >> 4;
        // rounds of T 16-byte pieces.  shift >= 16 * T, so what a round overwrites was read by an earlier round:
        // one barrier per round, one register quad per thread.
        for (uint32_t p = tid; p < n16 + tid; p += T) {   // uniform trip count: p - tid < n16
            if (p < n16) {
                const uint4 v = *reinterpret_cast<const uint4*>(win + shift + 16 * p);
                *reinterpret_cast<uint4*>(win + 16 * p) = v;
            }
            __syncthreads();
        }
        bpos += (int32_t)shift;
    };
    // one output byte at entry position pos < cur: from the window when still there, else from HBM
    auto read_out = [&](int64_t pos) -> uint8_t {
        if (pos >= bpos) return win[(uint32_t)(pos - bpos)];
        const uintptr_t a = reinterpret_cast<uintptr_t>(oblk + pos);
        const uint32_t w = ldcg32(reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3));
        return (uint8_t)(w >> (8 * (a & 3)));
    };
    // append n bytes from HBM (raw blocks, long literal runs); stride 0 = one repeated byte
    auto emit_global = [&](const uint8_t* src, uint32_t n, uint32_t stride) {
        uint32_t done = 0;
        const uint32_t rep = stride ? 0u : 0x01010101u * src[0];
        __syncthreads();
        while (done < n) {
            const uint32_t chunk = n - done < C::STEP ? n - done : C::STEP;
            reserve(chunk);
            uint8_t* d = win + (uint32_t)(cur - bpos);
            uint32_t head = (16u - ((uint32_t)(cur - bpos) & 15u)) & 15u;
            if (head > chunk) head = chunk;
            if (tid < head) d[tid] = stride ? src[done + tid] : (uint8_t)rep;
            const uint32_t body = (chunk - head) >> 4;     // 16-byte pieces into 16-byte aligned window rows
            for (uint32_t p = tid; p < body; p += T) {
                uint32_t w4[4] = {rep, rep, rep, rep};
                if (stride) load16_any(src + done + head + 16 * p, w4);
                *reinterpret_cast<uint4*>(d + head + 16 * p) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
            const uint32_t t0 = head + body * 16;
            if (t0 + tid < chunk) d[t0 + tid] = stride ? src[done + t0 + tid] : (uint8_t)rep;
            __syncthreads();
            cur += (int32_t)chunk; done += chunk;
            flush(false);
        }
    };
    // match copy of any length / offset (long matches), T bytes per round; off validated by the caller
    auto emit_match = [&](uint32_t off, uint32_t n) {
        uint32_t done = 0;
        __syncthreads();
        while (done < n) {
            const uint32_t m = n - done < T ? n - done : T;
            reserve(T);
            uint8_t v = 0;
            if (tid < m) {   // byte cur+tid repeats with period off: its source is the newest copy below cur
                const uint32_t k = tid < off ? 1u : tid / off + 1u;
                v = read_out((int64_t)cur + tid - (int64_t)off * k);
            }
            if (tid < m) win[(uint32_t)(cur - bpos) + tid] = v;   // sources are below cur: no overlap with this round's writes
            __syncthreads();
            cur += (int32_t)m; done += m;
            flush(false);
        }
    };

    int32_t fail = ST_OK;
    for (uint32_t k = blk_first; k < blk_end && fail == ST_OK; k++) {
        const ZBlock& b = blocks[k];
        // the prefix pass laid the blocks out back to back: this block starts where the previous one ended.  Rebase.
        oblk += cur; bpos -= cur; flushed -= cur; cur = 0;
        if (b.type == BT_RAW) { emit_global(buf + b.src, b.size, 1); continue; }
        if (b.type == BT_RLE) { emit_global(buf + b.src, b.size, 0); continue; }
        const uint8_t* lit;
        uint32_t lstride = 1;
        if (b.lit_type == LT_RAW) lit = buf + b.src + b.lit_pos;
        else if (b.lit_type == LT_RLE) { lit = buf + b.src + b.lit_pos; lstride = 0; }
        else lit = lits + zp->lit_base + b.lit_off;
        const uint32_t lit_regen = b.lit_regen, nseq = b.nseq;
        const SeqRec* sq = seqs + zp->seq_base + b.seq_off;
        const uint32_t rep_in[3] = {b.rep_in[0], b.rep_in[1], b.rep_in[2]};
        const uint64_t fd64 = b.out_off - b.frame_out;                // bytes of this frame before the block
        const uint32_t frame_dist = fd64 < 0x7FFFFFFFull ? (uint32_t)fd64 : 0x7FFFFFFFu;   // offsets beyond 2^31 are corrupt anyway
        uint32_t lp = 0;                                              // literals consumed
        uint32_t lit_loaded = 0;                                      // literal bytes staged so far (multiple of LIT_CH)
        __syncthreads();                                              // the previous block's last readers are done
        flush(false);
        if (!lstride) {                                               // RLE literals: the stage is that byte everywhere
            const uint8_t v = lit[0];
            for (uint32_t i = tid; i < C::LIT_RING + C::LIT_GUARD; i += T) lring[i] = v;
            lit_loaded = 0xFFFFFFFFu;
        }
        uint32_t staged = 0;                                          // sequence chunks issued so far
        // keep chunks c .. c+3 (c = wb / T) in flight; returns how many were issued now
        auto seq_issue = [&](uint32_t wb) -> uint32_t {
            const uint32_t c = wb / T;
            uint32_t issued = 0;
            while (staged <= c + 3 && staged * T < nseq) {
                const uint32_t i = staged * T + tid;
                if (i < nseq) cp_async8(sring + (staged & 3u) * T + tid, sq + i);
                cp_async_commit();
                staged++; issued++;
            }
            return issued;
        };
        // ---- registers of the NEXT step (its front runs one step ahead)
        uint32_t n_off = 1, n_ll = 0, n_ml = 0, n_dl = 0, n_sl = 0, n_nw = 0, n_ph = 0, n_incl = 0, n_llc = 0, n_totc = 0;
        uint32_t n_take = 0, n_wtot = 0, n_wlit = 0;                  // uniform
        uint32_t n_t[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        bool n_far = false, n_farc = false, n_bad = false;
        uint32_t n_start = 0;                                         // position where the next step begins
        auto front1 = [&](uint32_t wb) {
            const uint32_t i = wb + tid;
            const bool valid = i < nseq;
            SeqRec r{1u, 0u};
            if (valid) r = sring[((i / T) & 3u) * T + (i % T)];
            n_off = resolve_rep(r.x, rep_in);
            n_ll = r.y & 0xFFFFu; n_ml = r.y >> 16;
            bool longf = valid && (n_ll > LZ_SEQ_MAX || n_ml > LZ_SEQ_MAX);
            n_farc = valid && !longf && n_ml > 0 && n_off > C::KEEP;
            longf = longf || (n_farc && n_ml > LZ_FAR_MAX);
            n_llc = (valid && !longf) ? n_ll : 0u;
            n_totc = (valid && !longf) ? n_ll + n_ml : 0u;
            n_incl = warp_incl_scan((n_llc << 16) | n_totc, (int)lane);
            scan[warp * 32 + lane] = n_incl;
            const uint32_t stop = __ballot_sync(FULL, !valid || longf);
            if (lane == 0) wstop[warp] = stop ? (uint32_t)__ffs(stop) - 1u : 32u;
        };
        auto front2 = [&]() {
            // lane l stands for warp l: exclusive scan of the warp totals, first warp that holds the cut
            const uint32_t tv = lane < (uint32_t)C::W ? scan[lane * 32 + 31] : 0u;
            const uint32_t st_l = lane < (uint32_t)C::W ? wstop[lane] : 32u;
            const uint32_t tot_l = tv & 0xFFFFu, lit_l = tv >> 16;
            uint32_t bt = tot_l, bl = lit_l;
#pragma unroll
            for (int o = 1; o < C::W; o <<= 1) {
                const uint32_t x = __shfl_up_sync(FULL, bt, o), y = __shfl_up_sync(FULL, bl, o);
                if ((int)lane >= o) { bt += x; bl += y; }
            }
            bt -= tot_l; bl -= lit_l;                                  // exclusive
            const uint32_t fw = __ballot_sync(FULL, lane < (uint32_t)C::W && (st_l < 32u || bt + tot_l > C::STEP));
            uint32_t take, wtot, wlit;
            if (fw) {
                const uint32_t c = (uint32_t)__ffs(fw) - 1u;
                const uint32_t cbt = __shfl_sync(FULL, bt, c), cbl = __shfl_sync(FULL, bl, c), cst = __shfl_sync(FULL, st_l, c);
                const uint32_t v = scan[c * 32 + lane];
                const uint32_t fl = __ballot_sync(FULL, lane >= cst || cbt + (v & 0xFFFFu) > C::STEP);   // not empty
                const uint32_t f = (uint32_t)__ffs(fl) - 1u;
                const uint32_t pv = __shfl_sync(FULL, v, f ? f - 1 : 0);
                take = c * 32 + f;
                wtot = cbt + (f ? (pv & 0xFFFFu) : 0u);
                wlit = cbl + (f ? (pv >> 16) : 0u);
            } else {
                take = T;
                wtot = __shfl_sync(FULL, bt + tot_l, C::W - 1);
                wlit = __shfl_sync(FULL, bl + lit_l, C::W - 1);
            }
            const uint32_t my_bt = __shfl_sync(FULL, bt, warp), my_bl = __shfl_sync(FULL, bl, warp);
            n_take = take; n_wtot = wtot; n_wlit = wlit;
            const bool taken = tid < take;
            n_dl = my_bt + (n_incl & 0xFFFFu) - n_totc;               // step-relative start of this thread's literals
            n_sl = my_bl + (n_incl >> 16) - n_llc;                    // step-relative start in the literal stream
            const uint32_t dmp = n_start + n_dl + n_ll;               // position of the match
            n_bad = taken && (n_off == 0 || n_off > frame_dist + dmp);
            n_far = n_farc && taken && !n_bad;
            if (n_far) {   // the source has left (or will have left) the window; it is in HBM already: fetch it now
                const uintptr_t sp = reinterpret_cast<uintptr_t>(oblk + ((int64_t)dmp - (int64_t)n_off));
                const uint32_t* g = reinterpret_cast<const uint32_t*>(sp & ~(uintptr_t)3);
                n_nw = ((uint32_t)(sp & 3) + n_ml + 3) >> 2;          // <= 9 words
                n_ph = (uint32_t)(sp & 3);
#pragma unroll
                for (int q = 0; q < 9; q++) if ((uint32_t)q < n_nw) n_t[q] = ldcg32(g + q);
            }
        };
        bool any_bad = false;
        // full front for a step starting at sequence wb / entry position cur (block start, after a long sequence)
        auto prime = [&](uint32_t wb) {
            seq_issue(wb);
            cp_async_wait_all();
            __syncthreads();
            n_start = (uint32_t)cur;
            front1(wb);
            __syncthreads();
            front2();
            any_bad = __syncthreads_or(n_bad) != 0;
        };
        uint32_t wbase = 0;
        if (nseq) prime(0); else __syncthreads();
        while (wbase < nseq && fail == ST_OK) {
            // ---- take over the step prepared by the front
            const uint32_t off = n_off, ll = n_ll, ml = n_ml, dl = n_dl, sl = n_sl, wtot = n_wtot, wlit = n_wlit, ntake = n_take;
            const bool far = n_far;
            const uint32_t ph = n_ph;
            if (ntake == 0) {
                // the first sequence is long (or a long far match): it goes alone, by whole-CTA copies
                if (tid == 0) { misc[0] = off; misc[1] = ll; misc[2] = ml; }
                __syncthreads();
                const uint32_t o1 = misc[0];
                uint32_t l1 = misc[1], m1 = misc[2];
                if (l1 == SEQ_ESC || m1 == SEQ_ESC)
                    for (uint32_t q = 0; q < b.esc_n && q < (uint32_t)SEQ_ESC_MAX; q++)
                        if (b.esc_idx[q] == wbase) { l1 = b.esc_ll[q]; m1 = b.esc_ml[q]; }
                if ((uint64_t)lp + l1 > lit_regen) { fail = ST_INVALID_DATA; break; }
                if (l1) emit_global(lit + (size_t)lp * lstride, l1, lstride);
                lp += l1;
                if (o1 == 0 || o1 > frame_dist + (uint32_t)cur) { fail = ST_INVALID_DATA; break; }
                if (m1) emit_match(o1, m1);
                wbase += 1;
                if (wbase < nseq) prime(wbase); else __syncthreads();
                continue;
            }
            if (any_bad || (uint64_t)lp + wlit > lit_regen) { fail = ST_INVALID_DATA; break; }
            // ---- rows finished by the previous step; room in the window; the literals this step reads
            flush(false);
            reserve(C::STEP);
            if (lstride && lit_loaded < lp + wlit) {
                if (lit_loaded + C::LIT_RING < lp) lit_loaded = lp & ~(C::LIT_CH - 1);   // a long run was copied around the stage
                while (lit_loaded < lp + wlit) {
                    const uint32_t p = lit_loaded + 16 * tid;
                    if (16 * tid < C::LIT_CH && p < lit_regen) {      // 16-byte pieces, unaligned source
                        uint32_t w4[4];
                        load16_any(lit + p, w4);
                        const uint32_t si = p & (C::LIT_RING - 1);
                        const uint4 v = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                        *reinterpret_cast<uint4*>(lring + si) = v;
                        if (si < C::LIT_GUARD) *reinterpret_cast<uint4*>(lring + C::LIT_RING + si) = v;
                    }
                    lit_loaded += C::LIT_CH;
                }
            }
            const uint32_t step_start = (uint32_t)cur;               // >= 0 inside the block
            const uint32_t sidx = (uint32_t)(cur - bpos);            // window index of the step's first byte
            // ---- setup: source codes of this thread's bytes.  idx[] is indexed from the aligned window word that holds
            // the step's first byte (index = step-relative position + g0), so the resolve pass reads four codes per
            // 64-bit load and stores whole window words.
            const uint32_t g0 = sidx & 3u;
            if (tid < ntake) {
                Code* ix = idx + g0 + dl;
                fill_codes<Code>(ix, ll, (uint32_t)C::FLAG | (C::OFF_LIT + ((lp + sl) & (C::LIT_RING - 1))));   // guard covers the wrap
                ix += ll;
                if (far) {
                    // fetched during the previous step: the bytes go straight to their place, codes point at themselves.
                    // Source bytes ph.. of the fetched words -> destination bytes a.. of the aligned window words: one
                    // funnel shift per word; whole words are stored as words, the head and tail words byte-wise.
                    const uint32_t d = sidx + dl + ll;
                    const uint32_t a = d & 3u;
                    const int dlt = (int)ph - (int)a;
                    const uint32_t sh = (uint32_t)(dlt & 3) * 8u;
                    uint8_t* const wrow = win + (d - a);
                    const uint32_t end = a + ml;                          // row-relative end of the match
                    const uint32_t mt = end >> 2;                         // word that holds the tail (when end & 3)
                    uint32_t hw = 0, tw = 0;
#pragma unroll
                    for (int m = 0; m < 9; m++) {
                        const uint32_t lo_w = dlt < 0 ? (m ? n_t[m - 1] : 0u) : n_t[m];
                        const uint32_t hi_w = dlt < 0 ? n_t[m] : (m < 8 ? n_t[m + 1] : 0u);
                        const uint32_t wv = __funnelshift_r(lo_w, hi_w, sh);
                        if (m == 0) hw = wv;
                        if ((uint32_t)m == mt) tw = wv;
                        if ((m > 0 || a == 0) && 4u * m + 4u <= end) *reinterpret_cast<uint32_t*>(wrow + 4 * m) = wv;
                    }
                    if (a) {                                              // head word: bytes a .. min(3, end - 1)
#pragma unroll
                        for (uint32_t bb = 1; bb < 4; bb++) if (bb >= a && bb < end) wrow[bb] = (uint8_t)(hw >> (8 * bb));
                    }
                    if ((end & 3u) && (mt > 0 || a == 0)) {               // tail word: bytes 0 .. (end & 3) - 1
#pragma unroll
                        for (uint32_t bb = 0; bb < 3; bb++) if (bb < (end & 3u)) wrow[4 * mt + bb] = (uint8_t)(tw >> (8 * bb));
                    }
                    fill_codes<Code>(ix, ml, (uint32_t)C::FLAG | d);
                } else if (ml) {
                    const int32_t srel = (int32_t)(dl + ll) - (int32_t)off;             // step-relative source start
                    const uint32_t per = off < ml ? off : ml;                            // the match repeats with this period
                    const uint32_t nneg = srel < 0 ? ((uint32_t)(-srel) < per ? (uint32_t)(-srel) : per) : 0u;   // bytes that exist already
                    const uint32_t ecode = (uint32_t)C::FLAG | (uint32_t)((int32_t)sidx + srel);
                    const uint32_t scode = (uint32_t)((int32_t)g0 + srel);               // + q >= g0: produced by this step
                    fill_codes<Code>(ix, nneg, ecode);
                    fill_codes<Code>(ix + nneg, per - nneg, scode + nneg);
                    uint32_t r = 0;
                    for (uint32_t q = per; q < ml; q++) {                                // overlap: byte q equals byte q mod per
                        ix[q] = (Code)(r < nneg ? ecode + r : scode + r);
                        r = r + 1 == per ? 0u : r + 1;
                    }
                }
            }
            // ---- the next step's sequences (ring), per-warp scan
            wbase += ntake;
            const bool more = wbase < nseq;
            if (more) {
                const uint32_t issued = seq_issue(wbase);
                front1(wbase);
                if (issued == 1) cp_async_wait_1(); else cp_async_wait_all();
            }
            __syncthreads();
            // ---- resolve: byte-parallel; a thread takes one aligned window word (four bytes) per round, chases each
            // byte's code down to a byte that exists, and stores the word.  Bytes of the word outside the step (before its
            // start / behind its end) copy themselves.
            {
                constexpr uint32_t FL = (uint32_t)C::FLAG, M = FL - 1u;
                const uint32_t a0 = sidx - g0;                           // aligned window offset of idx[0]
                const uint32_t lim = g0 + wtot;
                const uint32_t ng = (lim + 3u) >> 2;
                for (uint32_t G = tid; G < ng; G += T) {
                    uint32_t c0, c1, c2, c3;
                    if constexpr (sizeof(Code) == 2) {
                        const uint2 cc = *reinterpret_cast<const uint2*>(idx + 4 * G);
                        c0 = cc.x & 0xFFFFu; c1 = cc.x >> 16; c2 = cc.y & 0xFFFFu; c3 = cc.y >> 16;
                    } else {
                        const uint4 cc = *reinterpret_cast<const uint4*>(idx + 4 * G);
                        c0 = cc.x; c1 = cc.y; c2 = cc.z; c3 = cc.w;
                    }
                    if (4 * G < g0 || 4 * G + 4 > lim) {                 // first / last word of the step
                        const uint32_t self = FL | (a0 + 4 * G);
                        if (4 * G + 0 < g0 || 4 * G + 0 >= lim) c0 = self;
                        if (4 * G + 1 < g0 || 4 * G + 1 >= lim) c1 = self + 1;
                        if (4 * G + 2 < g0 || 4 * G + 2 >= lim) c2 = self + 2;
                        if (4 * G + 3 < g0 || 4 * G + 3 >= lim) c3 = self + 3;
                    }
                    // The chase reads codes that other threads may be replacing at the same moment (path compression below):
                    // both sides use VOLATILE accesses of the code's own size, so a reader gets the old or the new code, never a
                    // torn one, and either leads to the same byte (codes strictly decrease along a chain).
                    volatile Code* const vidx = idx;
                    while (!((c0 & c1 & c2 & c3) & FL)) {
                        if (!(c0 & FL)) c0 = vidx[c0];
                        if (!(c1 & FL)) c1 = vidx[c1];
                        if (!(c2 & FL)) c2 = vidx[c2];
                        if (!(c3 & FL)) c3 = vidx[c3];
                    }
#ifndef PNA_LZ_NO_PATH_COMPRESSION
                    // path compression: later bytes of the step that chase into these stop after one hop
                    vidx[4 * G + 0] = (Code)c0; vidx[4 * G + 1] = (Code)c1; vidx[4 * G + 2] = (Code)c2; vidx[4 * G + 3] = (Code)c3;
#endif
                    const uint32_t v0 = lz_smem[c0 & M], v1 = lz_smem[c1 & M], v2 = lz_smem[c2 & M], v3 = lz_smem[c3 & M];
                    *reinterpret_cast<uint32_t*>(win + a0 + 4 * G) = v0 | (v1 << 8) | (v2 << 16) | (v3 << 24);
                }
            }
            if (more) { n_start = step_start + wtot; front2(); }
            cur = (int32_t)(step_start + wtot);
            lp += wlit;
            any_bad = __syncthreads_or(more && n_bad) != 0;
        }
        if (fail != ST_OK) break;
        // trailing literals of the block
        if (lp > lit_regen || (uint32_t)cur + (lit_regen - lp) != b.out_size) { fail = ST_INVALID_DATA; break; }
        if (lit_regen > lp) emit_global(lit + (size_t)lp * lstride, lit_regen - lp, lstride);
    }
    __syncthreads();
    if (fail == ST_OK) flush(true);
    if (fail != ST_OK && tid == 0) atomicCAS(&er.status, ST_OK, fail);
}

}  // namespace zs
}  // namespace pna
