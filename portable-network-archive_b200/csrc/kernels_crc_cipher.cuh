// kernels_crc_cipher.cuh -- sm_100a kernels: batched chunk CRC-32 (K1), AES-256 / Camellia-256
// CTR + CBC-decrypt + gather (K2/K3/K8), CBC-encrypt across entries, plain copies.
//
// All kernels are persistent-style: grid = a multiple of the SM count, CTAs loop over host-built
// tile tables, tables are staged into shared memory once per CTA.
#pragma once
#include <cuda_runtime.h>
#include <cstdlib>
#include "common.cuh"
#include "crc32_core.cuh"
#include "cipher_core.cuh"

namespace pna {

// ------------------------------------------------------------------------------------------------
// K1: CRC-32 of spans of a device image.  One warp per tile (<= CRC_TILE bytes).
struct CrcTile {
    uint64_t begin;   // byte offset in the image
    uint32_t len;     // <= CRC_TILE
    uint32_t span;    // which span this tile belongs to
};

// raw[t] = raw remainder (init 0, no xorout) of tile t
__global__ void __launch_bounds__(256) crc_tiles_kernel(const uint8_t* __restrict__ img, const CrcTile* __restrict__ tiles,
                                                        uint32_t n_tiles, const CrcConsts* __restrict__ C,
                                                        uint32_t* __restrict__ raw) {
    __shared__ uint32_t sU[CRC_NTAB * 256];
    __shared__ uint32_t sLane[32];
    __shared__ uint32_t sInv[16];
    for (int i = threadIdx.x; i < CRC_NTAB * 256; i += blockDim.x) sU[i] = (&C->U[0][0])[i];
    if (threadIdx.x < 32) sLane[threadIdx.x] = C->lane_k[threadIdx.x];
    if (threadIdx.x < 16) sInv[threadIdx.x] = C->inv_z[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warps_per_cta = blockDim.x >> 5;
    for (uint32_t t = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); t < n_tiles; t += gridDim.x * warps_per_cta) {
        const CrcTile tl = tiles[t];
        const uint64_t S = tl.begin, E = tl.begin + tl.len;
        const uint64_t A = (E + 15) & ~(uint64_t)15;
        const uint64_t rows = ((A - (S & ~(uint64_t)15)) + 511) / 512;
        uint32_t s = 0;
        int64_t a = (int64_t)A - (int64_t)rows * 512 + 16 * lane;   // oldest row first
        for (uint64_t r = 0; r < rows; r++, a += 512) {
            uint32_t w[4] = {0, 0, 0, 0};
            if (a + 16 > (int64_t)S && a < (int64_t)E && a >= 0) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(img + a));
                w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
                crc_mask_chunk((uint64_t)a, S, E, w);
            }
            s = crc_fold_row(s, w[0], w[1], w[2], w[3], sU);
        }
        uint32_t x = crc_multmodp(s, sLane[lane]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
        if (lane == 0) raw[t] = crc_multmodp(x, sInv[(16 - (E & 15)) & 15]);
    }
}

// The same tiles for batches large enough to fill the GPU: 1024 threads per CTA, one CTA per SM, and the four hot tables
// LANE-PRIVATE in shared memory ([table][byte][lane], 128 KB): lane l only ever touches bank l, so the 32 lookups of a warp
// instruction never conflict (the 1 KB tables of crc_tiles_kernel cost 3.1 wavefronts per lookup: random bytes, 32 lanes, 32
// banks).  The recurrence is also cheaper: a lane keeps FOUR registers, one per word of its 16-byte column, in the basis where
// a step is  s_j <- F(s_j ^ w_j),  F = "feed four bytes, then 508 zeros" -- four lookups per word, sixteen per 16 bytes (the
// 20-table form spends four more on advancing a separate state).  The last row is not advanced: s_j ^ w_j is the lane's
// 16-byte column remainder input, folded once per tile with the ordinary sixteen tables (from L1), then the lane constant,
// the XOR tree and the pad correction exactly as above.
constexpr int CRC_WIDE_THREADS = 1024;
constexpr int CRC_WIDE_SMEM = 4 * 256 * 32 * 4;
__global__ void __launch_bounds__(CRC_WIDE_THREADS, 1) crc_tiles_wide_kernel(const uint8_t* __restrict__ img, const CrcTile* __restrict__ tiles,
                                                                             uint32_t n_tiles, const CrcConsts* __restrict__ C,
                                                                             uint32_t* __restrict__ raw) {
    extern __shared__ uint32_t s_priv[];   // [k][b][lane] = U_{508+k}[b]
    for (int i = threadIdx.x; i < 4 * 256 * 32; i += blockDim.x) s_priv[i] = C->U[16 + (i >> 13)][(i >> 5) & 255];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t* const tl0 = s_priv + lane;   // + 32 * byte + 8192 * table
    const uint32_t* const U = &C->U[0][0];
    const uint32_t warps_per_cta = blockDim.x >> 5;
    // s ^ w advanced by 512 bytes: byte 0 of the word is the oldest (table U_511), byte 3 the newest (U_508)
    auto step = [&](uint32_t v) -> uint32_t {
        return tl0[3 * 8192 + ((v & 0xFFu) << 5)] ^ tl0[2 * 8192 + ((v >> 3) & 0x1FE0u)] ^ tl0[1 * 8192 + ((v >> 11) & 0x1FE0u)] ^
               tl0[0 * 8192 + ((v >> 19) & 0x1FE0u)];
    };
    for (uint32_t t = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); t < n_tiles; t += gridDim.x * warps_per_cta) {
        const CrcTile tl = tiles[t];
        const uint64_t S = tl.begin, E = tl.begin + tl.len;
        const uint64_t A = (E + 15) & ~(uint64_t)15;
        const uint32_t rows = (uint32_t)(((A - (S & ~(uint64_t)15)) + 511) / 512);
        uint32_t s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        int64_t a = (int64_t)A - (int64_t)rows * 512 + 16 * lane;   // oldest row first
        auto load_row = [&](int64_t at, uint32_t w[4]) {
            w[0] = w[1] = w[2] = w[3] = 0;
            if (at + 16 > (int64_t)S && at < (int64_t)E && at >= 0) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(img + at));
                w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
                crc_mask_chunk((uint64_t)at, S, E, w);
            }
        };
        uint32_t r = 0;
        // rows strictly inside the tile need no masking: four loads in flight per lane
        for (; r + 4 < rows; r += 4, a += 2048) {
            uint32_t w[4][4];
            if (r == 0) load_row(a, w[0]);
            else { const uint4 q = __ldg(reinterpret_cast<const uint4*>(img + a)); w[0][0] = q.x; w[0][1] = q.y; w[0][2] = q.z; w[0][3] = q.w; }
#pragma unroll
            for (int k = 1; k < 4; k++) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(img + a + 512 * k));
                w[k][0] = q.x; w[k][1] = q.y; w[k][2] = q.z; w[k][3] = q.w;
            }
#pragma unroll
            for (int k = 0; k < 4; k++) { s0 = step(s0 ^ w[k][0]); s1 = step(s1 ^ w[k][1]); s2 = step(s2 ^ w[k][2]); s3 = step(s3 ^ w[k][3]); }
        }
        for (; r + 1 < rows; r++, a += 512) {
            uint32_t w[4];
            load_row(a, w);
            s0 = step(s0 ^ w[0]); s1 = step(s1 ^ w[1]); s2 = step(s2 ^ w[2]); s3 = step(s3 ^ w[3]);
        }
        uint32_t x = 0;
        if (rows) {
            uint32_t w[4];
            load_row(a, w);
            x = crc_fold_row(0u, s0 ^ w[0], s1 ^ w[1], s2 ^ w[2], s3 ^ w[3], U);   // the column as 16 bytes, no advance
        }
        x = crc_multmodp(x, C->lane_k[lane]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
        if (lane == 0) raw[t] = crc_multmodp(x, C->inv_z[(16 - (E & 15)) & 15]);
    }
}
// tiles of a batch: the wide kernel once there is enough work to pay for its table fill on every SM
static inline void launch_crc_tiles(cudaStream_t stream, int sm_count, const uint8_t* img, const CrcTile* tiles, uint32_t nt, const CrcConsts* C,
                                    uint32_t* raw) {
    static const uint32_t wide_min = [] { const char* e = getenv("PNA_CRC_WIDE_MIN"); return e ? (uint32_t)strtoul(e, nullptr, 10) : 512u; }();
    if (nt >= wide_min) {   // every SM takes part; warps per CTA follow the work (4 .. 32)
        const uint32_t warps = std::min<uint32_t>(32u, std::max<uint32_t>(4u, (nt + (uint32_t)sm_count - 1) / (uint32_t)sm_count));
        const uint32_t grid = std::min<uint32_t>((nt + warps - 1) / warps, (uint32_t)sm_count);
        crc_tiles_wide_kernel<<<grid, 32 * warps, CRC_WIDE_SMEM, stream>>>(img, tiles, nt, C, raw);
    } else {
        const uint32_t grid = std::min<uint32_t>((nt + 7) / 8, (uint32_t)sm_count * 8);
        crc_tiles_kernel<<<grid, 256, 0, stream>>>(img, tiles, nt, C, raw);
    }
}

// combine the tiles of each span: acc <- acc * x^(8 len) ^ raw ; crc = ~acc
__global__ void crc_combine_kernel(const CrcTile* __restrict__ tiles, const uint32_t* __restrict__ raw,
                                   const uint32_t* __restrict__ span_first_tile, uint32_t n_spans, uint32_t n_tiles,
                                   const CrcConsts* __restrict__ C, uint32_t* __restrict__ crc_out,
                                   uint32_t init = 0xFFFFFFFFu /* register before the span: ~crc of a prefix (e.g. "FDAT") */) {
    uint32_t sp = blockIdx.x * blockDim.x + threadIdx.x;
    if (sp >= n_spans) return;
    uint32_t t0 = span_first_tile[sp], t1 = sp + 1 < n_spans ? span_first_tile[sp + 1] : n_tiles;
    uint32_t acc = init;
    for (uint32_t t = t0; t < t1; t++) {
        uint32_t len = tiles[t].len;
        uint32_t sh = len == CRC_TILE ? C->x_tile : crc_x2nmodp(C->x2n, len, 3);
        acc = crc_multmodp(sh, acc) ^ raw[t];
    }
    crc_out[sp] = ~acc;
}

// ------------------------------------------------------------------------------------------------
// Stream gather helpers.  An entry's stream is the concatenation of its segments.
__device__ __forceinline__ uint32_t find_segment(const Segment* segs, uint32_t n, uint64_t pos) {
    uint32_t lo = 0, hi = n;   // last segment with seg.pos <= pos
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (segs[mid].pos <= pos) lo = mid; else hi = mid;
    }
    return lo;
}
// 16 bytes from an arbitrary (unaligned) device address; the buffer is padded so over-reading the
// enclosing aligned words is safe.
__device__ __forceinline__ void load16_any(const uint8_t* p, uint32_t w[4]) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
    if (sh == 0) {
        if ((a & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(q);
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        } else { w[0] = q[0]; w[1] = q[1]; w[2] = q[2]; w[3] = q[3]; }
        return;
    }
    uint32_t t0 = q[0], t1 = q[1], t2 = q[2], t3 = q[3], t4 = q[4];
    w[0] = __funnelshift_r(t0, t1, sh); w[1] = __funnelshift_r(t1, t2, sh);
    w[2] = __funnelshift_r(t2, t3, sh); w[3] = __funnelshift_r(t3, t4, sh);
}
// 16 stream bytes starting at stream position `pos` (pos+16 <= stream_len), any segmentation
__device__ __forceinline__ void load_stream16(const uint8_t* buf, const Segment* segs, uint32_t n_segs,
                                              uint64_t stream_len, uint64_t pos, uint32_t w[4]) {
    uint32_t si = n_segs > 1 ? find_segment(segs, n_segs, pos) : 0;
    uint64_t seg_end = si + 1 < n_segs ? segs[si + 1].pos : stream_len;
    if (pos + 16 <= seg_end) {
        load16_any(buf + segs[si].img_off + (pos - segs[si].pos), w);
        return;
    }
    w[0] = w[1] = w[2] = w[3] = 0;
    for (int k = 0; k < 16; k++) {   // straddles bodies (IV or a block split across FDAT chunks)
        uint64_t p = pos + k;
        while (si + 1 < n_segs && segs[si + 1].pos <= p) si++;
        uint32_t b = buf[segs[si].img_off + (p - segs[si].pos)];
        w[k >> 2] |= b << (8 * (k & 3));
    }
}
__device__ __forceinline__ uint8_t load_stream1(const uint8_t* buf, const Segment* segs, uint32_t n_segs, uint64_t pos) {
    uint32_t si = n_segs > 1 ? find_segment(segs, n_segs, pos) : 0;
    return buf[segs[si].img_off + (pos - segs[si].pos)];
}

// ------------------------------------------------------------------------------------------------
// K2/K3/K8: decrypt (or plain gather) tiles of entry streams into the comp arena.
struct CipherTile {
    uint32_t entry;
    uint32_t n_blocks;     // 16-byte blocks in this tile (the last one of a CTR stream may be partial)
    uint64_t first_block;  // block index inside the entry's ciphertext (after the IV)
};
constexpr uint32_t CIPHER_TILE_BLOCKS = 1024;   // 16 KiB per tile

struct DevKeys {   // one per distinct (cipher, key)
    uint32_t aes_rk[60];
    uint32_t aes_dk[60];
    uint64_t cam_ek[34];
    uint64_t cam_dk[34];
};

// dynamic shared memory layout: [AES table 256*32 u32 (replicated)] or [Camellia sp_hi|sp_lo 2*2048 u32],
// then per-CTA key words.  256 threads per CTA.  AES-CTR has its own kernel (aes_ctr_tiles_kernel).
template <int ENC /*1 aes, 2 camellia, 0 none*/, int MODE /*0 cbc, 1 ctr*/>
__global__ void __launch_bounds__(256) decrypt_tiles_kernel(uint8_t* __restrict__ buf, const Segment* __restrict__ segs,
                                                            EntryRec* __restrict__ entries,
                                                            const CipherTile* __restrict__ tiles, uint32_t n_tiles,
                                                            const DevKeys* __restrict__ keys,
                                                            const AesTables* __restrict__ aes,
                                                            const CamelliaTables* __restrict__ cam) {
    static_assert(!(ENC == 1 && MODE == 1), "AES-CTR runs aes_ctr_tiles_kernel");
    extern __shared__ uint32_t smem[];
    uint32_t* s_tab = smem;
    uint8_t* s_isb = nullptr;
    if (ENC == 1) {
        const uint32_t* src = aes->td0;
        for (int i = threadIdx.x; i < 256 * 32; i += blockDim.x) s_tab[i] = src[i >> 5];   // [x*32 + lane]
        s_isb = reinterpret_cast<uint8_t*>(smem + 256 * 32);
        if (MODE == 0) for (int i = threadIdx.x; i < 256; i += blockDim.x) s_isb[i] = aes->inv_sbox[i];
    } else if (ENC == 2) {
        for (int i = threadIdx.x; i < 2048; i += blockDim.x) {
            s_tab[i] = (&cam->sp_hi[0][0])[i];
            s_tab[2048 + i] = (&cam->sp_lo[0][0])[i];
        }
    }
    __shared__ uint32_t s_key32[60];
    __shared__ uint64_t s_key64[34];
    __shared__ int s_key_idx;
    if (threadIdx.x == 0) s_key_idx = -2;
    __syncthreads();
    const TabView tv{s_tab, 32, (uint32_t)(threadIdx.x & 31)};

    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const CipherTile tl = tiles[t];
        const EntryRec e = entries[tl.entry];
        const Segment* sg = segs + e.seg_begin;
        if (ENC != 0 && e.key_idx != s_key_idx) {   // (re)load round keys for this tile's entry
            __syncthreads();
            const DevKeys* k = keys + e.key_idx;
            if (ENC == 1) { if (threadIdx.x < 60) s_key32[threadIdx.x] = k->aes_dk[threadIdx.x]; }
            else { if (threadIdx.x < 34) s_key64[threadIdx.x] = MODE == 1 ? k->cam_ek[threadIdx.x] : k->cam_dk[threadIdx.x]; }
            if (threadIdx.x == 0) s_key_idx = e.key_idx;
            __syncthreads();
        }
        const uint64_t hdr = ENC ? 16 : 0;               // IV prefix
        const uint64_t clen = e.stream_len - hdr;        // ciphertext bytes
        uint32_t iv[4] = {0, 0, 0, 0};
        if (ENC) load_stream16(buf, sg, e.n_segs, e.stream_len, 0, iv);
        uint8_t* dst = buf + e.comp_off;
        for (uint32_t j = threadIdx.x; j < tl.n_blocks; j += blockDim.x) {
            const uint64_t bi = tl.first_block + j;
            const uint64_t pos = hdr + bi * 16;
            const uint32_t have = (uint32_t)(clen - bi * 16 >= 16 ? 16 : clen - bi * 16);
            uint32_t c[4] = {0, 0, 0, 0};
            if (have == 16) load_stream16(buf, sg, e.n_segs, e.stream_len, pos, c);
            else for (uint32_t k = 0; k < have; k++) c[k >> 2] |= (uint32_t)load_stream1(buf, sg, e.n_segs, pos + k) << (8 * (k & 3));
            uint32_t o[4];
            if (ENC == 0) { o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = c[3]; }
            else if (MODE == 1) {   // CTR: keystream = E(IV + bi)
                ctr128be_add(iv, bi, o);
                camellia256_crypt_block(o, s_key64, s_tab, s_tab + 2048);
                o[0] ^= c[0]; o[1] ^= c[1]; o[2] ^= c[2]; o[3] ^= c[3];
            } else {                // CBC: P = D(C_i) ^ C_{i-1}
                uint32_t prev[4];
                if (bi == 0) { prev[0] = iv[0]; prev[1] = iv[1]; prev[2] = iv[2]; prev[3] = iv[3]; }
                else load_stream16(buf, sg, e.n_segs, e.stream_len, pos - 16, prev);
                o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = c[3];
                if (ENC == 1) aes256_decrypt_block(o, s_key32, tv, s_isb);
                else camellia256_crypt_block(o, s_key64, s_tab, s_tab + 2048);
                o[0] ^= prev[0]; o[1] ^= prev[1]; o[2] ^= prev[2]; o[3] ^= prev[3];
                if ((bi + 1) * 16 == clen) {   // last block: PKCS#7 unpad (cipher/block/read.rs:101)
                    uint32_t pad = o[3] >> 24;
                    bool ok = pad >= 1 && pad <= 16;
                    if (ok)
                        for (uint32_t k = 16 - pad; k < 16; k++) ok = ok && (((o[k >> 2] >> (8 * (k & 3))) & 0xFF) == pad);
                    if (ok) entries[tl.entry].comp_len = clen - pad;
                    else { entries[tl.entry].comp_len = 0; atomicCAS(&entries[tl.entry].status, ST_OK, ST_INVALID_DATA); }
                }
            }
            if (have == 16) *reinterpret_cast<uint4*>(dst + bi * 16) = make_uint4(o[0], o[1], o[2], o[3]);
            else for (uint32_t k = 0; k < have; k++) dst[bi * 16 + k] = (uint8_t)(o[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// AES-256-CTR extract.  A tile is a contiguous piece of ONE body (the host cuts tiles at body boundaries) and carries what a
// block would otherwise look up: its image offset, its destination and the counter block of its first block.  A tile spans
// at most CTR_TILE_RUNS counter runs (aes256_ctr_run_init), one per warp: lane l of warp w takes the blocks of run w whose
// counter low byte is l, l + 32, .., l + 224 -- up to 8 blocks that share the run's rounds 1-2, contiguous across the warp so
// that loads and stores coalesce.  A block that straddles two bodies is a tile of its own (src == CTR_TILE_SLOW), gathered
// through the entry's segments.
struct CtrTile {
    uint64_t src;       // image offset of the first ciphertext byte, or CTR_TILE_SLOW
    uint64_t dst;       // arena offset of the first output byte (16-byte aligned)
    uint32_t ctr[4];    // counter block of the first block (IV + block index), words as loaded
    uint32_t n_bytes;   // ciphertext bytes (the entry's last block may be partial)
    uint32_t key_idx;
    uint32_t entry;     // CTR_TILE_SLOW: whose segments to gather from ...
    uint32_t _pad;
    uint64_t pos;       // ... starting at this stream position
};
constexpr uint64_t CTR_TILE_SLOW = ~(uint64_t)0;
constexpr uint32_t CTR_TILE_RUNS = 32;                 // = warps per CTA
constexpr int AES_CTR_THREADS = 1024;                  // one CTA per SM: the tables take 128 KB
constexpr int AES_CTR_SMEM = AES_TE4_WORDS * 4 + 256;  // the create kernel keeps its keys in static shared memory
constexpr int AES_CTR_TILES_SMEM = AES_TE4_WORDS * 4 + CTR_TILE_RUNS * 64 * 4;   // + each warp's round keys
// n <= 16 stream bytes at stream position pos of entry *e, any segmentation (kept out of the kernel's hot loop)
__device__ __noinline__ uint4 ctr_gather_block(const uint8_t* buf, const Segment* segs, const EntryRec* e, uint64_t pos, uint32_t n) {
    uint32_t w[4] = {0, 0, 0, 0};
    if (n == 16) { load_stream16(buf, segs + e->seg_begin, e->n_segs, e->stream_len, pos, w); return make_uint4(w[0], w[1], w[2], w[3]); }
    uint64_t lo = 0, hi = 0;   // no register array indexed at run time: it would go to local memory
    for (uint32_t k = 0; k < n; k++) {
        const uint64_t v = load_stream1(buf, segs + e->seg_begin, e->n_segs, pos + k);
        if (k < 8) lo |= v << (8 * k); else hi |= v << (8 * (k - 8));
    }
    return make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
}
__global__ void __launch_bounds__(AES_CTR_THREADS, 1) aes_ctr_tiles_kernel(uint8_t* __restrict__ buf, const Segment* __restrict__ segs,
                                                                           const EntryRec* __restrict__ entries,
                                                                           const CtrTile* __restrict__ tiles, uint32_t n_tiles,
                                                                           const DevKeys* __restrict__ keys,
                                                                           const AesTables* __restrict__ aes) {
    extern __shared__ __align__(16) uint32_t smem[];
    aes_te4_fill(smem, aes);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* const s_rk = smem + AES_TE4_WORDS + 64 * warp;
    __syncthreads();
    const LaneTe4 t{reinterpret_cast<const uint8_t*>(smem), lane * 4};
    const uint32_t* const rk = static_cast<const uint32_t*>(__builtin_assume_aligned(s_rk, 16));
    uint32_t have_key = 0xFFFFFFFFu;
    for (uint32_t ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const CtrTile tl = tiles[ti];
        const uint32_t n_blocks = (tl.n_bytes + 15) / 16;
        const int32_t j0 = (int32_t)(256 * warp) - (int32_t)(tl.ctr[3] >> 24);   // tile block of this run's low byte 0
        if (j0 + 256 <= 0 || j0 >= (int32_t)n_blocks) continue;                  // the tile has no block in run `warp`
        if (tl.key_idx != have_key) {
            __syncwarp();
            for (uint32_t i = lane; i < 60; i += 32) s_rk[i] = keys[tl.key_idx].aes_rk[i];
            have_key = tl.key_idx;
            __syncwarp();
        }
        uint32_t run[4] = {tl.ctr[0], tl.ctr[1], tl.ctr[2], tl.ctr[3] & 0x00FFFFFFu};
        ctr128be_add(run, 256u * warp, run);   // carries through all 128 bits and wraps at 2^128
        uint32_t p[5];
        aes256_ctr_run_init(run, rk, t, p);

        const bool slow = tl.src == CTR_TILE_SLOW;
        const uintptr_t sa = reinterpret_cast<uintptr_t>(buf) + (slow ? 0 : tl.src);
        const uint4* const q = reinterpret_cast<const uint4*>(sa & ~(uintptr_t)15);   // aligned 16-byte words of the tile
        const uint32_t wo = (uint32_t)(sa >> 2) & 3, sh = (uint32_t)(sa & 3) * 8;
        // ciphertext of tile block j: the enclosing aligned 16 bytes and the next, then a funnel shift (bodies are not aligned)
        auto load = [&](int32_t j, uint32_t c[4]) {
            if (slow) {
                const uint4 v = ctr_gather_block(buf, segs, entries + tl.entry, tl.pos, tl.n_bytes);
                c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
                return;
            }
            const uint4 a = __ldg(q + j);
            const uint4 b = (sa & 15) ? __ldg(q + j + 1) : make_uint4(0, 0, 0, 0);
            uint32_t v0, v1, v2, v3, v4;
            switch (wo) {
                case 0: v0 = a.x; v1 = a.y; v2 = a.z; v3 = a.w; v4 = b.x; break;
                case 1: v0 = a.y; v1 = a.z; v2 = a.w; v3 = b.x; v4 = b.y; break;
                case 2: v0 = a.z; v1 = a.w; v2 = b.x; v3 = b.y; v4 = b.z; break;
                default: v0 = a.w; v1 = b.x; v2 = b.y; v3 = b.z; v4 = b.w; break;
            }
            c[0] = __funnelshift_r(v0, v1, sh); c[1] = __funnelshift_r(v1, v2, sh);
            c[2] = __funnelshift_r(v2, v3, sh); c[3] = __funnelshift_r(v3, v4, sh);
        };
        auto in_tile = [&](int32_t j) { return j >= 0 && j < (int32_t)n_blocks; };
        uint8_t* const dst = buf + tl.dst;
        uint32_t c[4] = {0, 0, 0, 0};
        if (in_tile(j0 + (int32_t)lane)) load(j0 + (int32_t)lane, c);
#pragma unroll 1
        for (uint32_t x = lane; x < 256; x += 32) {
            const int32_t j = j0 + (int32_t)x;
            uint32_t cn[4] = {0, 0, 0, 0};
            if (x + 32 < 256 && in_tile(j + 32)) load(j + 32, cn);   // the keystream does not wait for the data
            if (in_tile(j)) {
                uint32_t o[4];
                aes256_ctr_run_block(p, x << 24, rk, t, o);
                o[0] ^= c[0]; o[1] ^= c[1]; o[2] ^= c[2]; o[3] ^= c[3];
                const uint32_t have = tl.n_bytes - 16 * (uint32_t)j;
                if (have >= 16) *reinterpret_cast<uint4*>(dst + 16 * (uint32_t)j) = make_uint4(o[0], o[1], o[2], o[3]);
                else {
                    const uint64_t lo = o[0] | (uint64_t)o[1] << 32, hi = o[2] | (uint64_t)o[3] << 32;
                    for (uint32_t k = 0; k < have; k++) dst[16 * (uint32_t)j + k] = (uint8_t)(k < 8 ? lo >> (8 * k) : hi >> (8 * (k - 8)));
                }
            }
            c[0] = cn[0]; c[1] = cn[1]; c[2] = cn[2]; c[3] = cn[3];
        }
    }
}

// ECB test hook (KATs lib/src/cipher.rs:256-292 are CBC of one block == ECB(pt ^ iv))
__global__ void ecb_kernel(int enc, int encrypt, const DevKeys* __restrict__ key, const AesTables* __restrict__ aes,
                           const CamelliaTables* __restrict__ cam, const uint8_t* __restrict__ in, uint64_t n_blocks,
                           uint8_t* __restrict__ out) {
    extern __shared__ uint32_t smem[];
    uint32_t* s_tab = smem;
    uint8_t* s_isb = reinterpret_cast<uint8_t*>(smem + 256 * 32);
    if (enc == 1) {
        const uint32_t* src = encrypt ? aes->te0 : aes->td0;
        for (int i = threadIdx.x; i < 256 * 32; i += blockDim.x) s_tab[i] = src[i >> 5];
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_isb[i] = aes->inv_sbox[i];
    } else {
        for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_tab[i] = (&cam->sp_hi[0][0])[i]; s_tab[2048 + i] = (&cam->sp_lo[0][0])[i]; }
    }
    __syncthreads();
    const TabView tv{s_tab, 32, (uint32_t)(threadIdx.x & 31)};
    for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < n_blocks; b += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t s[4];
        load16_any(in + b * 16, s);
        if (enc == 1) { if (encrypt) aes256_encrypt_block(s, key->aes_rk, tv); else aes256_decrypt_block(s, key->aes_dk, tv, s_isb); }
        else camellia256_crypt_block(s, encrypt ? key->cam_ek : key->cam_dk, s_tab, s_tab + 2048);
        for (int k = 0; k < 16; k++) out[b * 16 + k] = (uint8_t)(s[k >> 2] >> (8 * (k & 3)));
    }
}

// ------------------------------------------------------------------------------------------------
// plain device copy of many (dst,src,len) jobs: one warp per 4 KiB piece (store entries, gathers)
struct CopyJob { uint64_t dst, src, len; };
__global__ void copy_jobs_kernel(uint8_t* __restrict__ dst_base, const uint8_t* __restrict__ src_base,
                                 const CopyJob* __restrict__ jobs, uint32_t n_jobs) {
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n_jobs; j += warps) {
        const CopyJob c = jobs[j];
        uint8_t* d = dst_base + c.dst;
        const uint8_t* s = src_base + c.src;
        if ((((uintptr_t)d | (uintptr_t)s) & 15) == 0) {
            uint64_t v = c.len / 16;
            for (uint64_t i = lane; i < v; i += 32) reinterpret_cast<uint4*>(d)[i] = reinterpret_cast<const uint4*>(s)[i];
            for (uint64_t i = v * 16 + lane; i < c.len; i += 32) d[i] = s[i];
        } else {
            for (uint64_t i = lane; i < c.len; i += 32) d[i] = s[i];
        }
    }
}

}  // namespace pna
