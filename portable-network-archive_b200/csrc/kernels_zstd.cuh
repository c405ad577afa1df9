// kernels_zstd.cuh -- sm_100a kernels for zstd frame decode (K4).  See zstd_core.cuh for the format
// logic and DESIGN.md for the phase plan:
//   zstd_count/fill  (thread per entry)  frame + block header walk
//   zstd_parse       (thread per block)  literal/sequence section headers, table description offsets
//   zstd_resolve     (thread per entry)  Repeat_Mode / treeless sources, per-entry literal+sequence offsets
//   zstd_order       (one CTA)           counting sort of the blocks by sequence / literal count (load balance)
//   zstd_seq         (LANE per block)    FSE sequence decode; 32 blocks per warp, 16-bit tables interleaved in smem
//   zstd_lit         (lane per stream)   Huffman literals, 8 blocks x 4 streams per warp, tables in smem
//   zstd_prefix      (thread per entry)  output offsets, absolute repeat-offset history per block
//   zstd_lz          (CTA per entry)     LZ execution in a shared-memory window, 32*W sequences per step (kernels_zstd_lz.cuh)
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"
#include "zstd_core.cuh"
#include "kernels_crc_cipher.cuh"   // load16_any
#include "kernels_zstd_lz.cuh"       // ZEntry, zstd_lz_kernel<LzSmall|LzBig>
#include "kernels_zstd_pj.cuh"       // block-parallel LZ inside one frame (pointer jumping)

namespace pna {
namespace zs {

__device__ __forceinline__ void set_status(EntryRec* entries, uint32_t e, int32_t st) {
    if (st != ST_OK) atomicCAS(&entries[e].status, ST_OK, st);
}

__global__ void zstd_count_kernel(const uint8_t* __restrict__ buf, EntryRec* entries, ZEntry* ze, uint32_t nz) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nz) return;
    const uint32_t e = ze[i].entry;
    uint32_t nb = 0;
    int32_t st = ST_OK;
    if (entries[e].status == ST_OK) st = scan_entry(buf, entries[e].comp_off, entries[e].comp_len, e, nullptr, &nb);
    set_status(entries, e, st);
    ze[i].blk_count = st == ST_OK && entries[e].status == ST_OK ? nb : 0;
}
// Re-walks the frames (the entry table is reset at the start of every run, so the status has to be re-established here
// too).  The walk is serial per entry -- a block is found only behind the previous block's header -- so it records 16 bytes
// per block; zstd_fill_kernel builds the ZBlock records with a thread per block.
__global__ void zstd_walk_kernel(const uint8_t* __restrict__ buf, EntryRec* entries, const ZEntry* ze, uint32_t nz,
                                 WalkRec* __restrict__ walk) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nz) return;
    const uint32_t e = ze[i].entry;
    if (entries[e].status != ST_OK) return;
    uint32_t nb = 0;
    int32_t st = scan_entry(buf, entries[e].comp_off, entries[e].comp_len, e, nullptr, &nb, walk + ze[i].blk_begin, ze[i].blk_count);
    if (st == ST_OK && nb != ze[i].blk_count) st = ST_INTERNAL;
    set_status(entries, e, st);
}
__global__ void zstd_fill_kernel(const EntryRec* __restrict__ entries, const WalkRec* __restrict__ walk, uint32_t n_blocks, ZBlock* blocks) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_blocks) return;
    const WalkRec w = walk[i];
    ZBlock z;
    zblock_from_walk(w, z);
    if (entries[w.entry].status != ST_OK) z.status = ST_INTERNAL;   // the walk failed: nothing of this entry is decoded
    blocks[i] = z;
}
__global__ void zstd_parse_kernel(const uint8_t* __restrict__ buf, EntryRec* entries, ZBlock* blocks, uint32_t n_blocks) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_blocks) return;
    ZBlock b = blocks[i];
    b.status = parse_block(buf, b);
    blocks[i] = b;
    set_status(entries, b.entry, b.status);
}
// value of a "last writer wins" variable as lane `lane` sees it (its own write included): the newest writer at or below the
// lane, else the value carried in from the previous chunk
__device__ __forceinline__ int32_t last_writer(uint32_t writers, int32_t myval, int32_t carry, uint32_t lane) {
    const uint32_t m = writers & (0xFFFFFFFFu >> (31u - lane));
    const int src = m ? 31 - __clz((int)m) : 0;
    const int32_t v = __shfl_sync(0xFFFFFFFFu, myval, src);
    return m ? v : carry;
}
// Repeat_Mode / treeless sources, literal and sequence offsets, frame count of every entry (zstd_core.cuh resolve_sources,
// restated as warp scans: ONE WARP per entry, 32 blocks per round -- a solid archive is one entry of tens of thousands of
// blocks, which a thread per entry would walk for tens of milliseconds).
__global__ void __launch_bounds__(128) zstd_resolve_kernel(EntryRec* entries, ZEntry* ze, uint32_t nz, ZBlock* blocks) {
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
    if (i >= nz) return;
    const ZEntry z = ze[i];
    uint64_t lit = 0, seq = 0;
    uint32_t nf = 0;
    if (entries[z.entry].status == ST_OK) {
        int32_t c_huf = -2, c_cur[3] = {-2, -2, -2};
        bool bad = false;
        for (uint32_t k0 = z.blk_begin; k0 < z.blk_begin + z.blk_count; k0 += 32) {
            const uint32_t k = k0 + lane;
            const bool have = k < z.blk_begin + z.blk_count;
            ZBlock* b = blocks + (have ? k : k0);
            const bool first = have && b->first_in_frame;
            const bool comp = have && b->type == BT_COMPRESSED;
            const bool live = comp && b->status == ST_OK;                  // resolve_sources skips the others
            const uint32_t lt = b->lit_type, nseq = b->nseq, lit_regen = b->lit_regen;
            // Huffman tree source
            {
                const bool own = live && lt == LT_COMPRESSED;
                const uint32_t w = __ballot_sync(0xFFFFFFFFu, first || own);
                const int32_t seen = last_writer(w, own ? (int32_t)k : -2, c_huf, lane);
                if (live) { if (lt == LT_TREELESS && seen < 0) bad = true; b->huf_src = seen; }
                c_huf = __shfl_sync(0xFFFFFFFFu, last_writer(w, own ? (int32_t)k : -2, c_huf, 31u), 31);
            }
#pragma unroll
            for (int t = 0; t < 3; t++) {
                const uint32_t mode = b->mode[t];
                const bool uses = live && nseq != 0;
                const bool own = uses && mode != SM_REPEAT;
                const int32_t val = own ? (mode == SM_PREDEF ? -1 : (int32_t)k) : -2;
                const uint32_t w = __ballot_sync(0xFFFFFFFFu, first || own);
                const int32_t seen = last_writer(w, val, c_cur[t], lane);
                if (uses) { if (mode == SM_REPEAT && seen == -2) bad = true; b->tsrc[t] = seen; }
                c_cur[t] = __shfl_sync(0xFFFFFFFFu, last_writer(w, val, c_cur[t], 31u), 31);
            }
            // literal / sequence arena offsets (exclusive sums), relative to the entry's bases
            const uint32_t lc = (comp && lt >= LT_COMPRESSED) ? ((lit_regen + 15u) & ~15u) : 0u, sc = comp ? nseq : 0u;
            const uint32_t li = warp_incl_scan(lc, (int)lane), si = warp_incl_scan(sc, (int)lane);
            if (have) { b->lit_off = lit + li - lc; b->seq_off = seq + si - sc; }
            lit += __shfl_sync(0xFFFFFFFFu, li, 31);
            seq += __shfl_sync(0xFFFFFFFFu, si, 31);
            nf += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, first));
        }
        if (__any_sync(0xFFFFFFFFu, bad) && lane == 0) set_status(entries, z.entry, ST_INVALID_DATA);
    }
    if (lane == 0) { ze[i].lit_total = lit; ze[i].seq_total = seq; ze[i].n_frames = nf; }
}
// LZ units of every entry: one per frame, in stream order, at the entry's slots (ZEntry.unit_begin from the host)
__global__ void zstd_units_kernel(const ZEntry* __restrict__ ze, uint32_t nz, const ZBlock* __restrict__ blocks, LzUnit* __restrict__ units) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nz) return;
    const ZEntry z = ze[i];
    const uint32_t u = z.unit_begin;
    uint32_t made = 0;
    for (uint32_t k = z.blk_begin; k < z.blk_begin + z.blk_count; k++) {
        if (blocks[k].first_in_frame && made < z.n_frames) { units[u + made] = LzUnit{i, k, 0u, 0u}; made++; }
        if (made) units[u + made - 1].blk_count++;
    }
}

// ------------------------------------------------------------------------------------------------
// Block ordering: blocks with sequences sorted by descending sequence count (so the 32 lanes of a warp
// of zstd_seq_kernel finish together), blocks with Huffman literals by descending literal count.
// counts[0] = sequence blocks, counts[1] = literal blocks, counts[2..3] = work counters (zeroed here).
__global__ void __launch_bounds__(1024) zstd_order_kernel(const EntryRec* __restrict__ entries, const ZBlock* __restrict__ blocks,
                                                          uint32_t n_blocks, uint32_t* __restrict__ seq_order,
                                                          uint32_t* __restrict__ lit_order, uint32_t* __restrict__ counts) {
    __shared__ uint32_t hs[1024], hl[1024];
    __shared__ uint32_t carry[2];
    const uint32_t tid = threadIdx.x;
    hs[tid] = 0; hl[tid] = 0;
    __syncthreads();
    auto keys = [&](uint32_t i, uint32_t& ks, uint32_t& kl) {
        const ZBlock& b = blocks[i];
        ks = kl = 0xFFFFFFFFu;
        if (b.type != BT_COMPRESSED || b.status != ST_OK || entries[b.entry].status != ST_OK) return;
        if (b.nseq > 0) { uint32_t k = b.nseq >> 6; ks = 1023u - (k > 1023u ? 1023u : k); }
        if (b.lit_type >= LT_COMPRESSED) { uint32_t k = b.lit_regen >> 7; kl = 1023u - (k > 1023u ? 1023u : k); }
    };
    for (uint32_t i = tid; i < n_blocks; i += 1024) {
        uint32_t ks, kl;
        keys(i, ks, kl);
        if (ks != 0xFFFFFFFFu) atomicAdd(&hs[ks], 1u);
        if (kl != 0xFFFFFFFFu) atomicAdd(&hl[kl], 1u);
    }
    __syncthreads();
    // exclusive scan of both histograms (1024 bins, one per thread): warp scan + warp totals
    uint32_t vs = hs[tid], vl = hl[tid];
    const int lane = tid & 31, warp = tid >> 5;
    uint32_t is = vs, il = vl;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t a = __shfl_up_sync(0xFFFFFFFFu, is, o), b = __shfl_up_sync(0xFFFFFFFFu, il, o);
        if (lane >= o) { is += a; il += b; }
    }
    __shared__ uint32_t ws[32], wl[32];
    if (lane == 31) { ws[warp] = is; wl[warp] = il; }
    __syncthreads();
    if (warp == 0) {
        uint32_t a = ws[lane], b = wl[lane], ia = a, ib = b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t x = __shfl_up_sync(0xFFFFFFFFu, ia, o), y = __shfl_up_sync(0xFFFFFFFFu, ib, o);
            if (lane >= o) { ia += x; ib += y; }
        }
        ws[lane] = ia - a; wl[lane] = ib - b;
        if (lane == 31) { carry[0] = ia; carry[1] = ib; }
    }
    __syncthreads();
    hs[tid] = ws[warp] + is - vs;
    hl[tid] = wl[warp] + il - vl;
    __syncthreads();
    for (uint32_t i = tid; i < n_blocks; i += 1024) {
        uint32_t ks, kl;
        keys(i, ks, kl);
        if (ks != 0xFFFFFFFFu) seq_order[atomicAdd(&hs[ks], 1u)] = i;
        if (kl != 0xFFFFFFFFu) lit_order[atomicAdd(&hl[kl], 1u)] = i;
    }
    if (tid == 0) { counts[0] = carry[0]; counts[1] = carry[1]; counts[2] = 0; counts[3] = 0; counts[4] = 0; }
}

// ------------------------------------------------------------------------------------------------
// Sequence stage.  The FSE chain (table lookup -> bit counts -> next state) is serial per block, so throughput = blocks in
// flight / chain latency, and blocks in flight = shared memory / table bytes: 16-bit cells (zstd_core.cuh Tab16) make a
// block's three tables 2.5 KB, 88 blocks fill the SM's 227 KB.  One CTA of 4 warps per SM (one warp per scheduler), 22 table
// sets per warp, interleaved by set; the warps take batches of 22 blocks independently (no CTA barrier).
// Measured dead end (round 2, profiles/r2_seq_streams_per_lane.txt): advancing K independent blocks per lane (22 / K lanes
// active) to fill the empty issue slots takes K times as long -- 9.7 / 17.9 / 25.8 ms for K = 1 / 2 / 3 on the cfg2 shard.
// The kernel is not waiting on latency that a second chain could fill: with ONE warp per scheduler the integer pipe issues
// a warp instruction every two cycles at best, the loop runs at 0.27 of a possible 0.5 IPC, and fewer active lanes per warp
// means more warp instructions for the same sequences.  What would help is fewer instructions per sequence or smaller tables.
// Fewer instructions (profiles/r3_seq_ab.log): the common path of the step loop is 112 static SASS instructions (73 ALU-pipe,
// 22 IMAD, 10 memory, 7 control), against 184 before (110 / 45 / 11 / 17), and the stage went from 9.5 to 7.4 ms on the cfg2
// shard (one B200, 1000 W limit, 1965 MHz).  The rare paths (second window, ring refill, escapes) are not counted.
constexpr uint32_t SEQ_SLOTS = 22, SEQ_WARPS = 4;
constexpr uint32_t SEQ_TAB_BYTES = TAB16_TOTAL * SEQ_SLOTS * SEQ_WARPS * sizeof(uint16_t);    // 225280
constexpr uint32_t SEQ_SMEM_BYTES = SEQ_TAB_BYTES + SEQ_SLOTS * SEQ_WARPS * 64;               // + a 64-byte bitstream ring per block in flight

// A lane's bitstream through shared memory: 16 words (four 16-byte groups) of the stream around the read position,
// refilled one group at a time by cp.async two groups before it is needed.  The stream is consumed downwards at
// <= 3 words per window, so one conditional refill per window keeps groups (A>>2) and (A>>2)-1 resident and complete.
struct RingBitSrc {
    uint32_t* ring;            // this lane's 16 words (64-byte aligned shared memory)
    uint32_t rs;               // its shared-memory address: word k of the ring is at rs | (k & 15) * 4
    const uint32_t* words;     // arena start: nothing below it is fetched
    const uint32_t* gbase;     // 16-byte aligned group that holds the stream's first byte
    int32_t qoff;              // bit index from gbase of the bit below position 0: position p's top bit is p + qoff
    int32_t gl;                // lowest group loaded or in flight
    __device__ __forceinline__ void fetch(int32_t g) {
        const uint32_t* src = gbase + 4 * (int64_t)g;
        if (src >= words) {
            cp_async16(ring + ((uint32_t)g & 3u) * 4u, src);
            cp_async_commit();
        } else cp_async_wait_all();   // nothing newer will follow: drain
    }
    __device__ __forceinline__ void init(const uint32_t* w, uint64_t begin, int32_t pos) {
        words = w;
#if defined(PNA_EMU)
        rs = 0;
#else
        rs = (uint32_t)__cvta_generic_to_shared(ring);
#endif
        const uint32_t* wb = w + (begin >> 2);
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(wb) >> 2) & 3u;   // word phase of the start in its group
        gbase = wb - mis;
        qoff = (int32_t)(mis * 32 + (uint32_t)(begin & 3) * 8) - 1;
        gl = ((pos + qoff) >> 7) - 3;
        for (int32_t g = gl + 3; g >= gl; g--) fetch(g);
        cp_async_wait_all();
    }
    __device__ __forceinline__ uint64_t window(int32_t pos) {
        const int32_t q = pos + qoff;                     // bit index from gbase of the window's top bit (>= -1)
        const uint32_t o = (uint32_t)q >> 3;              // bits 2-5: ring byte offset of the window's top word
        const uint32_t sh = ~(uint32_t)q & 31u;
        if ((q >> 7) <= gl + 2) { gl--; fetch(gl); }
        cp_async_wait_1();
        const uint32_t h = word(o), m = word(o - 4u), l = word(o - 8u);
        return ((uint64_t)__funnelshift_l(m, h, sh) << 32) | __funnelshift_l(l, m, sh);
    }
    // the ring word at byte offset o mod 64: one LOP3 for the address, since the ring is 64-byte aligned
    __device__ __forceinline__ uint32_t word(uint32_t o) const {
#if defined(PNA_EMU)
        return ring[(o & 60u) >> 2];
#else
        uint32_t v;   // volatile: stays behind the cp.async wait that makes the word visible
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(rs | (o & 60u)));
        return v;
#endif
    }
};
__global__ void __launch_bounds__(32 * SEQ_WARPS) zstd_seq_kernel(const uint8_t* __restrict__ buf, EntryRec* entries, ZBlock* blocks,
                                                                  const uint32_t* __restrict__ order, uint32_t* counts,
                                                                  const uint64_t* __restrict__ seq_base_of_entry,
                                                                  SeqRec* __restrict__ seqs) {
    extern __shared__ __align__(64) uint16_t stab_all[];
    __shared__ uint32_t s_llb[36], s_mlb[53];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c = threadIdx.x; c < 36; c += blockDim.x) s_llb[c] = seq_pack_ll((uint32_t)c);
    for (int c = threadIdx.x; c < 53; c += blockDim.x) s_mlb[c] = seq_pack_ml((uint32_t)c);
    __syncthreads();
    const uint32_t n = counts[0];
    const uint32_t* words = reinterpret_cast<const uint32_t*>(buf);
    uint16_t* const stab = stab_all + (uint32_t)warp * TAB16_TOTAL * SEQ_SLOTS;
    const bool active = (uint32_t)lane < SEQ_SLOTS;
    const uint32_t slot = active ? (uint32_t)lane : 0u;
    const Tab16 tll{stab + TAB16_LL * SEQ_SLOTS + slot, SEQ_SLOTS}, tml{stab + TAB16_ML * SEQ_SLOTS + slot, SEQ_SLOTS},
        tof{stab + TAB16_OF * SEQ_SLOTS + slot, SEQ_SLOTS};
    for (;;) {
        uint32_t first = 0;
        if (lane == 0) first = atomicAdd(&counts[2], SEQ_SLOTS);
        first = __shfl_sync(0xFFFFFFFFu, first, 0);
        if (first >= n) break;
        const uint32_t k = first + (uint32_t)lane;
        if (active && k < n) {
            ZBlock& gb = blocks[order[k]];
            int16_t norm[64];
            uint16_t next_of[64];
            const int l0 = seq_tab16_for(buf, blocks, gb, 0, tll, norm, next_of);
            const int l1 = seq_tab16_for(buf, blocks, gb, 1, tof, norm, next_of);
            const int l2 = seq_tab16_for(buf, blocks, gb, 2, tml, norm, next_of);
            int32_t st = ST_INVALID_DATA;
            if (l0 >= 0 && l1 >= 0 && l2 >= 0) {
                SeqStream<RingBitSrc> s;   // scalars only: lives in registers (no L1 is left beside 225 KB of tables)
                s.src.ring = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(stab_all) + SEQ_TAB_BYTES) + ((uint32_t)warp * SEQ_SLOTS + slot) * 16;
                st = s.begin(words, buf, gb, tll, tof, tml, l0, l1, l2, s_llb, s_mlb, seqs + seq_base_of_entry[gb.entry] + gb.seq_off);
                if (st == ST_OK) {
                    const uint32_t nseq = s.nseq;
                    for (uint32_t i = 0; i < nseq; i++) s.step(i);
                    st = s.end();
                }
            }
            if (st != ST_OK) { gb.status = st; set_status(entries, gb.entry, st); }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// Literal stage: one lane per Huffman stream, 8 blocks (x4 streams) per warp; each block's single-symbol
// table (<= 8 KB at the format's maximum log 12) sits in shared memory and is shared by its 4 lanes.
constexpr uint32_t LIT_SLOTS = 8;
constexpr uint32_t LIT_SMEM_BYTES = LIT_SLOTS * (1u << HUF_LOG_MAX) * sizeof(uint16_t);   // 65536
__global__ void __launch_bounds__(32) zstd_lit_kernel(const uint8_t* __restrict__ buf, EntryRec* entries, ZBlock* blocks,
                                                      const uint32_t* __restrict__ order, uint32_t* counts,
                                                      const uint64_t* __restrict__ lit_base_of_entry, uint8_t* __restrict__ lits) {
    extern __shared__ uint16_t shuf[];
    __shared__ int s_log[LIT_SLOTS], s_hdr[LIT_SLOTS];
    const int lane = threadIdx.x, slot = lane >> 2, sub = lane & 3;
    const uint32_t n = counts[1];
    const uint32_t* words = reinterpret_cast<const uint32_t*>(buf);
    uint16_t* table = shuf + slot * (1u << HUF_LOG_MAX);
    for (;;) {
        uint32_t batch = 0;
        if (lane == 0) batch = atomicAdd(&counts[3], 1u);
        batch = __shfl_sync(0xFFFFFFFFu, batch, 0);
        if ((uint64_t)batch * LIT_SLOTS >= n) break;
        const uint32_t k = batch * LIT_SLOTS + slot;
        const bool have = k < n;
        const uint32_t bi = have ? order[k] : 0;
        if (have && sub == 0) {
            const ZBlock& gb = blocks[bi];
            const ZBlock& hb = blocks[gb.huf_src];
            uint8_t weights[260];
            FseEntry wfse[64];
            int hlog = 0;
            const int hdr = huf_read_table(words, buf, hb.src + hb.lit_pos, hb.lit_csize, table, &hlog, weights, wfse);
            s_log[slot] = hlog; s_hdr[slot] = hdr;
        }
        __syncwarp();
        if (have) {
            ZBlock& gb = blocks[bi];
            bool ok = s_hdr[slot] >= 0;
            const uint32_t lit_csize = gb.lit_csize, lit_regen = gb.lit_regen;
            const uint32_t skip = gb.lit_type == LT_COMPRESSED ? (uint32_t)(ok ? s_hdr[slot] : 0) : 0;
            if (ok && skip > lit_csize) ok = false;
            const uint64_t at = gb.src + gb.lit_pos + skip;
            const uint32_t clen = lit_csize - (ok ? skip : 0);
            uint8_t* dst = lits + lit_base_of_entry[gb.entry] + gb.lit_off;
            if (ok) {
                if (gb.lit_streams == 1) {
                    if (sub == 0) ok = huf_decode_stream_w(words, buf, at, clen, table, s_log[slot], dst, lit_regen);
                } else {
                    uint32_t s1 = 0, s2 = 0, s3 = 0;
                    if (clen < 6) ok = false;
                    else { s1 = load_le16(buf + at); s2 = load_le16(buf + at + 2); s3 = load_le16(buf + at + 4); }
                    if (ok && (uint64_t)s1 + s2 + s3 + 6 > clen) ok = false;
                    const uint32_t seg = (lit_regen + 3) / 4;
                    if (ok && seg * 3 > lit_regen) ok = false;
                    if (ok) {
                        const uint32_t sz = sub == 0 ? s1 : sub == 1 ? s2 : sub == 2 ? s3 : clen - 6 - s1 - s2 - s3;
                        const uint64_t o = at + 6 + (sub > 0 ? s1 : 0) + (sub > 1 ? s2 : 0) + (sub > 2 ? s3 : 0);
                        const uint32_t cnt = sub < 3 ? seg : lit_regen - 3 * seg;
                        ok = huf_decode_stream_w(words, buf, o, sz, table, s_log[slot], dst + (uint64_t)sub * seg, cnt);
                    }
                }
            }
            if (!ok) { atomicCAS(&gb.status, ST_OK, ST_INVALID_DATA); set_status(entries, gb.entry, ST_INVALID_DATA); }
        }
        __syncwarp();
    }
}

// Output offsets, frame starts and the absolute incoming repeat-offset history of every block (zstd_core.cuh prefix_entry):
// ONE WARP per entry, 32 blocks per round -- positions by warp scans, the history by a register-only walk over the 32
// blocks' (symbolic) outgoing histories, so that no round waits on memory more than once.
__global__ void __launch_bounds__(128) zstd_prefix_kernel(EntryRec* entries, const ZEntry* ze, uint32_t nz, ZBlock* blocks) {
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
    if (i >= nz) return;
    const ZEntry z = ze[i];
    if (entries[z.entry].status != ST_OK) return;
    uint64_t pos = 0, frame_start = 0;
    uint32_t rep[3] = {1, 4, 8};
    int32_t st = ST_OK;
    for (uint32_t k0 = z.blk_begin; k0 < z.blk_begin + z.blk_count; k0 += 32) {
        const uint32_t k = k0 + lane;
        const bool have = k < z.blk_begin + z.blk_count;
        ZBlock* b = blocks + (have ? k : k0);
        const bool first = have && b->first_in_frame;
        const int32_t bst = have ? b->status : ST_OK;
        const bool ok = have && bst == ST_OK;
        const uint32_t osz = ok ? b->out_size : 0u;                       // a failed block does not advance (prefix_entry)
        const bool upd = ok && b->type == BT_COMPRESSED && b->nseq > 0;
        const uint32_t ro0 = b->rep_out[0], ro1 = b->rep_out[1], ro2 = b->rep_out[2];
        const uint32_t incl = warp_incl_scan(osz, (int)lane);
        const uint64_t my_pos = pos + incl - osz;
        // frame start = position of the newest first_in_frame block at or below this one
        const uint32_t fw = __ballot_sync(0xFFFFFFFFu, first);
        const uint32_t fm = fw & (0xFFFFFFFFu >> (31u - lane));
        const uint32_t fsrc = fm ? 31u - (uint32_t)__clz((int)fm) : 0u;
        const uint32_t fpos_lo = __shfl_sync(0xFFFFFFFFu, (uint32_t)my_pos, (int)fsrc), fpos_hi = __shfl_sync(0xFFFFFFFFu, (uint32_t)(my_pos >> 32), (int)fsrc);
        const uint64_t my_frame = fm ? (((uint64_t)fpos_hi << 32) | fpos_lo) : frame_start;
        // repeat-offset history: every lane walks the 32 blocks in registers, lane j keeps what block j sees
        uint32_t in0 = 0, in1 = 0, in2 = 0;
        int32_t my_st = bst;
        for (int j = 0; j < 32; j++) {
            const bool jf = (fw >> j) & 1u;
            if (jf) { rep[0] = 1; rep[1] = 4; rep[2] = 8; }
            if ((int)lane == j) { in0 = rep[0]; in1 = rep[1]; in2 = rep[2]; }
            const bool ju = __shfl_sync(0xFFFFFFFFu, upd ? 1 : 0, j) != 0;
            const uint32_t a0 = __shfl_sync(0xFFFFFFFFu, ro0, j), a1 = __shfl_sync(0xFFFFFFFFu, ro1, j), a2 = __shfl_sync(0xFFFFFFFFu, ro2, j);
            if (ju) {
                const uint32_t r0 = resolve_rep(a0, rep), r1 = resolve_rep(a1, rep), r2 = resolve_rep(a2, rep);
                if (!r0 || !r1 || !r2) { if ((int)lane == j) my_st = ST_INVALID_DATA; }
                else { rep[0] = r0; rep[1] = r1; rep[2] = r2; }
            }
        }
        if (have) {
            b->out_off = my_pos; b->frame_out = my_frame;
            b->rep_in[0] = in0; b->rep_in[1] = in1; b->rep_in[2] = in2;
            if (my_st != bst) b->status = my_st;
        }
        // first failure in block order (a failed entry produces no output, so the positions behind it do not matter)
        const uint32_t badm = __ballot_sync(0xFFFFFFFFu, have && my_st != ST_OK);
        const int32_t first_bad = __shfl_sync(0xFFFFFFFFu, my_st, badm ? __ffs((int)badm) - 1 : 0);
        if (badm && st == ST_OK) st = first_bad;
        pos += __shfl_sync(0xFFFFFFFFu, incl, 31);
        const int fl = fw ? 31 - __clz((int)fw) : 0;
        const uint32_t fs_lo = __shfl_sync(0xFFFFFFFFu, (uint32_t)my_pos, fl), fs_hi = __shfl_sync(0xFFFFFFFFu, (uint32_t)(my_pos >> 32), fl);
        if (fw) frame_start = ((uint64_t)fs_hi << 32) | fs_lo;
    }
    if (lane == 0) {
        set_status(entries, z.entry, st);
        entries[z.entry].out_len = pos;
    }
}

}  // namespace zs
}  // namespace pna
