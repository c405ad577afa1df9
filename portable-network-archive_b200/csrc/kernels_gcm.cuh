// kernels_gcm.cuh -- sm_100a kernels of the GCM STREAM cipher mode (cipher mode 2; reference lib/src/cipher/gcm.rs:206-290
// decrypt reader, :44-63 encrypt writer; lib/src/cipher/aead.rs:92-150,210-217 header and segment nonce).
//
// A data stream is header(75) || { ciphertext(<= segment_size) || tag(16) } per segment.  Segments are independent
// (own nonce), and inside a segment both halves of GCM are data-parallel:
//   * CTR: keystream block j = E_K(nonce || BE32(2 + j)) -- the same counter walk as the CTR kernels;
//   * GHASH: Y = sum C_i * H^(n-i), evaluated per 16 KiB tile by ONE WARP: lane l takes the blocks l, l+32, l+64, ... of the
//     tile (coalesced 512-byte rows, the same 16 bytes feed the hash and the keystream XOR) with a Horner step of H^32, the 32
//     lane values are folded by a 5-level tree with H, H^2, ..., H^16, and the tiles of a segment are chained with H^1024 by the
//     finishing kernel, which also adds the length block, E_K(J0) and compares (or writes) the tag.
// The first tile of a segment is the short one, so every later tile is a full 1024 blocks and the chain needs one power only.
// Per key the setup kernel derives H = E_K(0) and the seven power tables (gcm_core.cuh); keys are per entry (HKDF of the entry
// header, aead.rs:188), so this is per entry work.
#pragma once
#include <cuda_runtime.h>
#include "kernels_crc_cipher.cuh"
#include "gcm_core.cuh"

namespace pna {
namespace gcm {

constexpr uint32_t GCM_HEADER_LEN = 75, GCM_TAG_LEN = 16, GCM_MAX_SEGMENT = 67108864u;
constexpr uint32_t GCM_TILE_BLOCKS = 1024;   // 16 KiB per warp task

struct GcmSeg {           // one segment of one entry; self-contained, so the decode and the encode plan share the kernels
    uint32_t entry;       // whose status a failed tag sets
    uint32_t pow_idx;     // which GcmPow (one per GCM entry of the plan)
    uint32_t nonce[3];    // the 12 nonce bytes as loaded (little-endian words)
    uint32_t first_tile, n_tiles;
    int32_t key_idx;      // round keys
    uint32_t enc;         // 1 AES-256, 2 Camellia-256
    uint32_t src_n_segs;  // the source stream: a list of bodies (decode) or of compressed pieces (encode) ...
    uint64_t src_seg_begin;
    uint64_t src_len;     // ... and its total length
    uint64_t ct_pos;      // position of this segment's bytes in the source stream
    uint64_t ct_len;      // ciphertext bytes; the tag follows them.  GCM_SEG_UNUSED: slot not used (encode plans are sized by bounds)
    uint64_t dst_off;     // where the segment's output goes in the destination buffer
};
constexpr uint64_t GCM_SEG_UNUSED = ~0ull;
struct GcmTile { uint32_t seg, n_blocks; uint64_t first_block; };   // n_blocks == 0: unused slot
struct GcmKeyRef { int32_t key_idx; uint32_t enc; };                // pow_idx -> key

__device__ __forceinline__ void block_encrypt(int enc, uint32_t s[4], const uint32_t* rk32, const uint64_t* rk64, const TabView& tv,
                                              const uint32_t* cam_hi, const uint32_t* cam_lo) {
    if (enc == 1) aes256_encrypt_block(s, rk32, tv);
    else camellia256_crypt_block(s, rk64, cam_hi, cam_lo);
}

// ------------------------------------------------------------------------------------------------
// per key: H and its power tables.  One thread per key; cipher tables unreplicated in shared memory.
__global__ void __launch_bounds__(128) gcm_setup_kernel(const GcmKeyRef* __restrict__ refs, uint32_t n, const DevKeys* __restrict__ keys, const AesTables* __restrict__ aes,
                                                        const CamelliaTables* __restrict__ cam, GcmPow* __restrict__ pows) {
    __shared__ uint32_t s_te[256];
    __shared__ uint32_t s_cam[4096];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_te[i] = aes->te0[i];
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_cam[i] = (&cam->sp_hi[0][0])[i]; s_cam[2048 + i] = (&cam->sp_lo[0][0])[i]; }
    __syncthreads();
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const GcmKeyRef r = refs[k];
    if (r.key_idx < 0) return;
    const DevKeys* dk = keys + r.key_idx;
    uint32_t s[4] = {0, 0, 0, 0};
    block_encrypt((int)r.enc, s, dk->aes_rk, dk->cam_ek, TabView{s_te, 1, 0}, s_cam, s_cam + 2048);
    make_powers(from_le_words(s[0], s[1], s[2], s[3]), pows + k);
}

// ------------------------------------------------------------------------------------------------
// tiles: CTR + partial GHASH.  ENC 1 AES-256, 2 Camellia-256.  The source is gathered through a Segment list (the entry's
// bodies on decode, the compressed pieces on encode); DECRYPT only decides which side of the XOR is hashed.
struct GcmWarpState {   // per-warp shared memory
    GTab t[GCM_N_POW];
    uint32_t rk32[60];
    uint64_t rk64[34];
};
// AES: the four rotations of Te0 as four lane-replicated tables (128 KB, no rotate per lookup -- two thirds of this kernel's
// instructions are AES) and 32 warps in ONE CTA per SM, like the CTR kernel; Camellia: 16 KB of SP tables, 8 warps, 3 CTAs per SM.
template <int ENC>
constexpr int gcm_tile_warps() { return ENC == 1 ? 32 : 8; }
template <int ENC>
constexpr int gcm_tiles_smem() { return (ENC == 1 ? 4 * 256 * 32 * 4 : 2 * 2048 * 4) + gcm_tile_warps<ENC>() * (int)sizeof(GcmWarpState) + 64; }

template <int ENC, bool DECRYPT>
__global__ void __launch_bounds__(gcm_tile_warps<ENC>() * 32) gcm_tiles_kernel(const uint8_t* __restrict__ src, const Segment* __restrict__ segs,
                                                                       uint8_t* __restrict__ dst_base,
                                                                       const GcmSeg* __restrict__ gsegs, const GcmTile* __restrict__ tiles,
                                                                       uint32_t n_tiles, const DevKeys* __restrict__ keys,
                                                                       const GcmPow* __restrict__ pows, const AesTables* __restrict__ aes,
                                                                       const CamelliaTables* __restrict__ cam,
                                                                       G128* __restrict__ partial) {
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* s_tab = smem;
    constexpr int TAB_WORDS = ENC == 1 ? 4 * 256 * 32 : 2 * 2048;
    constexpr int GCM_TILE_WARPS = ENC == 1 ? 32 : 8;
    GcmWarpState* ws_all = reinterpret_cast<GcmWarpState*>(smem + TAB_WORDS);
    uint32_t* s_last4 = reinterpret_cast<uint32_t*>(ws_all + GCM_TILE_WARPS);
    if (ENC == 1) aes_te4_fill(s_tab, aes);
    else for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_tab[i] = (&cam->sp_hi[0][0])[i]; s_tab[2048 + i] = (&cam->sp_lo[0][0])[i]; }
    if (threadIdx.x < 16) { const uint32_t l4[16] = PNA_GCM_LAST4; s_last4[threadIdx.x] = l4[threadIdx.x]; }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    GcmWarpState& ws = ws_all[warp];
    uint32_t have_pow = 0xFFFFFFFFu;
    const uint32_t n_warps = gridDim.x * GCM_TILE_WARPS;
    for (uint32_t t = blockIdx.x * GCM_TILE_WARPS + warp; t < n_tiles; t += n_warps) {
        const GcmTile tl = tiles[t];
        if (tl.n_blocks == 0) continue;
        const GcmSeg sg = gsegs[tl.seg];
        if (sg.pow_idx != have_pow) {   // this warp's key material
            __syncwarp();
            const uint32_t* ps = reinterpret_cast<const uint32_t*>(pows + sg.pow_idx);
            uint32_t* pd = reinterpret_cast<uint32_t*>(ws.t);
            for (uint32_t i = lane; i < sizeof(GcmPow) / 4; i += 32) pd[i] = ps[i];
            const DevKeys* dk = keys + sg.key_idx;
            if (ENC == 1) { for (uint32_t i = lane; i < 60; i += 32) ws.rk32[i] = dk->aes_rk[i]; }
            else for (uint32_t i = lane; i < 34; i += 32) ws.rk64[i] = dk->cam_ek[i];
            have_pow = sg.pow_idx;
            __syncwarp();
        }
        const Segment* bs = segs + sg.src_seg_begin;
        const uint32_t pad = GCM_TILE_BLOCKS - tl.n_blocks;   // the short tile is right-aligned: leading zero blocks
        G128 y = G128{{0, 0, 0, 0}};
        for (uint32_t k = pad >> 5; k < 32; k++) {
            const uint32_t r = k * 32 + lane;
            y = mul_table(y, ws.t[GCM_POW_STRIDE].e, s_last4);
            if (r < pad) continue;
            const uint64_t bi = tl.first_block + (r - pad);
            const uint64_t off = bi * 16;
            const uint32_t have = (uint32_t)(sg.ct_len - off >= 16 ? 16 : sg.ct_len - off);
            uint32_t c[4] = {0, 0, 0, 0};
            if (sg.ct_pos + off + 16 <= sg.src_len) load_stream16(src, bs, sg.src_n_segs, sg.src_len, sg.ct_pos + off, c);
            else for (uint32_t q = 0; q < have; q++) c[q >> 2] |= (uint32_t)load_stream1(src, bs, sg.src_n_segs, sg.ct_pos + off + q) << (8 * (q & 3));
            if (have < 16) {   // only this segment's bytes
                const uint32_t keep = have * 8;
                for (int q = 0; q < 4; q++) {
                    const uint32_t lo = q * 32;
                    if (keep <= lo) c[q] = 0; else if (keep < lo + 32) c[q] &= (1u << (keep - lo)) - 1u;
                }
            }
            uint32_t o[4] = {sg.nonce[0], sg.nonce[1], sg.nonce[2], bswap32((uint32_t)bi + 2u)};   // inc32 from J0 + 1
            if (ENC == 1) {
                aes256_encrypt_block4(o, ws.rk32, LaneTe4{reinterpret_cast<const uint8_t*>(s_tab), lane * 4});
            } else camellia256_crypt_block(o, ws.rk64, s_tab, s_tab + 2048);
            o[0] ^= c[0]; o[1] ^= c[1]; o[2] ^= c[2]; o[3] ^= c[3];
            if (!DECRYPT && have < 16) {   // the hash sees the ciphertext zero-padded
                const uint32_t keep = have * 8;
                for (int q = 0; q < 4; q++) {
                    const uint32_t lo = q * 32;
                    if (keep <= lo) o[q] = 0; else if (keep < lo + 32) o[q] &= (1u << (keep - lo)) - 1u;
                }
            }
            const uint32_t* hw = DECRYPT ? c : o;     // GHASH runs over the ciphertext
            G128 x = from_le_words(hw[0], hw[1], hw[2], hw[3]);
            gxor(y, x);
            uint8_t* dst = dst_base + sg.dst_off + off;
            if (have == 16 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
            else for (uint32_t q = 0; q < have; q++) dst[q] = (uint8_t)(o[q >> 2] >> (8 * (q & 3)));
        }
        // lanes -> tile: left half of every pair carries 2^l more blocks behind it
#pragma unroll 1
        for (int l = 0; l < 5; l++) {
            const G128 m = mul_table(y, ws.t[l].e, s_last4);
            if (!((lane >> l) & 1)) y = m;
            y.w[0] ^= __shfl_xor_sync(0xFFFFFFFFu, y.w[0], 1 << l);
            y.w[1] ^= __shfl_xor_sync(0xFFFFFFFFu, y.w[1], 1 << l);
            y.w[2] ^= __shfl_xor_sync(0xFFFFFFFFu, y.w[2], 1 << l);
            y.w[3] ^= __shfl_xor_sync(0xFFFFFFFFu, y.w[3], 1 << l);
        }
        if (lane == 0) partial[t] = mul_table(y, ws.t[0].e, s_last4);   // sum C_i H^(m-i), i = 0..m-1
    }
}

// ------------------------------------------------------------------------------------------------
// per segment: chain the tiles, add the length block, tag = GHASH ^ E_K(J0).  DECRYPT: compare with the stored tag
// (mismatch -> InvalidData, "authentication failed", gcm.rs:283); else write the tag behind the ciphertext.
template <bool DECRYPT>
__global__ void __launch_bounds__(128) gcm_finish_kernel(const uint8_t* __restrict__ src, const Segment* __restrict__ segs, EntryRec* __restrict__ entries,
                                                         const GcmSeg* __restrict__ gsegs, uint32_t n_segs, const DevKeys* __restrict__ keys,
                                                         const GcmPow* __restrict__ pows, const AesTables* __restrict__ aes,
                                                         const CamelliaTables* __restrict__ cam, const G128* __restrict__ partial,
                                                         uint8_t* __restrict__ dst_base) {
    __shared__ uint32_t s_te[256];
    __shared__ uint32_t s_cam[4096];
    __shared__ uint32_t s_last4[16];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_te[i] = aes->te0[i];
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) { s_cam[i] = (&cam->sp_hi[0][0])[i]; s_cam[2048 + i] = (&cam->sp_lo[0][0])[i]; }
    if (threadIdx.x < 16) { const uint32_t l4[16] = PNA_GCM_LAST4; s_last4[threadIdx.x] = l4[threadIdx.x]; }
    __syncthreads();
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_segs) return;
    const GcmSeg sg = gsegs[s];
    if (sg.ct_len == GCM_SEG_UNUSED) return;
    const GcmPow* pw = pows + sg.pow_idx;
    G128 y = G128{{0, 0, 0, 0}};
    for (uint32_t t = 0; t < sg.n_tiles; t++) {
        if (t) y = mul_table(y, pw->t[GCM_POW_TILE].e, s_last4);
        gxor(y, partial[sg.first_tile + t]);
    }
    const uint64_t bits = sg.ct_len * 8;       // len(A) = 0 || len(C)
    y.w[1] ^= (uint32_t)(bits >> 32); y.w[0] ^= (uint32_t)bits;
    y = mul_table(y, pw->t[0].e, s_last4);
    uint32_t j0[4] = {sg.nonce[0], sg.nonce[1], sg.nonce[2], bswap32(1u)};
    const DevKeys* dk = keys + sg.key_idx;
    block_encrypt((int)sg.enc, j0, dk->aes_rk, dk->cam_ek, TabView{s_te, 1, 0}, s_cam, s_cam + 2048);
    uint32_t tag[4];
    to_le_words(y, tag);
    tag[0] ^= j0[0]; tag[1] ^= j0[1]; tag[2] ^= j0[2]; tag[3] ^= j0[3];
    if (DECRYPT) {
        uint32_t got[4];
        load_stream16(src, segs + sg.src_seg_begin, sg.src_n_segs, sg.src_len, sg.ct_pos + sg.ct_len, got);
        if ((got[0] ^ tag[0]) | (got[1] ^ tag[1]) | (got[2] ^ tag[2]) | (got[3] ^ tag[3]))
            atomicCAS(&entries[sg.entry].status, ST_OK, ST_INVALID_DATA);
    } else {
        uint8_t* dst = dst_base + sg.dst_off + sg.ct_len;
        for (int q = 0; q < 16; q++) dst[q] = (uint8_t)(tag[q >> 2] >> (8 * (q & 3)));
    }
}

}  // namespace gcm
}  // namespace pna
