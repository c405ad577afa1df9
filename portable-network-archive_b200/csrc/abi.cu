// abi.cu -- C ABI of libpna_cuda.so (see include/pna_cuda.h): context, batch plans, host<->device
// staging and the kernel launch sequences for the PNA data-chunk pipeline on B200 (sm_100a).
//
// No CPU fallback lives here: every compute step is a kernel from kernels_*.cuh.  The host side
// only indexes (offsets, tiles, key schedules) and moves bytes.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pna_cuda.h"
#include "kernels_crc_cipher.cuh"
#include "kernels_gcm.cuh"
#include "aead_host.hpp"
#include "kernels_inflate.cuh"
#include "kernels_xz.cuh"
#include "kernels_zstd.cuh"
#include "kernels_encode.cuh"

using namespace pna;

// ------------------------------------------------------------------------------------------------
struct pna_ctx {
    // A context over several devices (pna_cuda_init with n_devices > 1) is a dispatcher: `devs` holds one single-device
    // context per GPU and every batch call shards its entries across them (multi_host.cuh).  Single-device contexts have no devs.
    std::vector<pna_ctx*> devs;
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t sync_ev = nullptr;   // blocking-sync event: waits sleep instead of spinning (many contexts per box share the host cores)
    std::mutex mu;
    std::string err;
    uint64_t launches = 0;
    std::vector<cudaEvent_t> ev_pool;   // stage-timing events, recycled between plans (no create/destroy per batch)
    CrcConsts* d_crc = nullptr;
    AesTables* d_aes = nullptr;
    CamelliaTables* d_cam = nullptr;
    AesTables h_aes;
    CamelliaTables h_cam;
    bool fail(const char* what, cudaError_t e) {
        err = std::string(what) + ": " + cudaGetErrorString(e);
        return false;
    }
    // wait for everything queued on the stream; the calling thread sleeps (cudaEventBlockingSync)
    cudaError_t sync() {
        cudaError_t e = cudaEventRecord(sync_ev, stream);
        return e == cudaSuccess ? cudaEventSynchronize(sync_ev) : e;
    }
};

#define CK(call)                                                       \
    do {                                                               \
        cudaError_t e__ = (call);                                      \
        if (e__ != cudaSuccess) { ctx->fail(#call, e__); return PNA_E_CUDA; } \
    } while (0)
#define LAUNCHED() do { ctx->launches++; CK(cudaGetLastError()); } while (0)

// Device memory cache: batch calls reuse the arenas of earlier calls instead of paying cudaMalloc/cudaFree
// (milliseconds for multi-GiB arenas) on every pna_cuda_decode_batch / encode_batch.
struct DevCache {
    struct Blk { void* p; size_t bytes; int dev; };
    std::mutex mu;
    std::vector<Blk> free_list;
    std::map<void*, std::pair<size_t, int>> live;
    std::map<int, cudaStream_t> alloc_streams;
    cudaStream_t alloc_stream(int dev) {
        std::lock_guard<std::mutex> g(mu);
        auto it = alloc_streams.find(dev);
        if (it != alloc_streams.end()) return it->second;
        cudaStream_t s = nullptr;
        cudaMemPool_t pool;
        uint64_t keep = UINT64_MAX;
        if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess || cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess ||
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep) != cudaSuccess) { cudaGetLastError(); s = nullptr; }
        alloc_streams[dev] = s;
        return s;
    }
    cudaError_t alloc(void** out, size_t bytes) {
        // size classes: 4 KiB steps below 64 KiB, 1 MiB up to 1 MiB, then quarter-octave steps (1, 1.25, 1.5, 1.75 x 2^k):
        // batches of similar shape ask for the SAME sizes, so a released arena is found again instead of a fresh cudaMalloc
        // (which stalls the calling worker behind every kernel in flight)
        if (bytes < ((size_t)64 << 10)) bytes = (bytes + 4095) & ~(size_t)4095;
        else if (bytes <= ((size_t)1 << 20)) bytes = (size_t)1 << 20;
        else {
            size_t k = 20;
            while (((size_t)2 << k) <= bytes) k++;          // 2^k <= bytes < 2^(k+1)
            const size_t step = ((size_t)1 << k) / 4;
            bytes = (bytes + step - 1) / step * step;
        }
        int dev = 0;
        cudaGetDevice(&dev);
        {
            std::lock_guard<std::mutex> g(mu);
            int best = -1;
            for (int i = 0; i < (int)free_list.size(); i++) {
                const Blk& b = free_list[i];
                if (b.dev != dev || b.bytes < bytes || b.bytes > bytes + bytes / 2 + ((size_t)4 << 20)) continue;
                if (best < 0 || b.bytes < free_list[best].bytes) best = i;
            }
            if (best >= 0) {
                *out = free_list[best].p;
                live[*out] = {free_list[best].bytes, dev};
                free_list.erase(free_list.begin() + best);
                return cudaSuccess;
            }
        }
        // the driver call runs outside the lock: other threads keep hitting the cache meanwhile
        // A miss goes to the stream-ordered allocator on a stream of its own: cudaMalloc waits for every kernel in flight on the
        // device (measured: 30-170 ms for a 1 MiB block in the middle of a pipelined extract), cudaMallocAsync does not, and the
        // pool keeps what it is given back (release threshold = everything).
        static const bool trace = getenv("PNA_HOST_TRACE") != nullptr;
        const auto t0 = std::chrono::steady_clock::now();
        cudaStream_t as = alloc_stream(dev);
        cudaError_t e = as ? cudaMallocAsync(out, bytes, as) : cudaMalloc(out, bytes);
        if (e == cudaSuccess && as) e = cudaStreamSynchronize(as);
        if (trace) fprintf(stderr, "[pna_cuda] device allocation (%zu MiB) took %.1f ms\n", bytes >> 20,
                           std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
        if (e != cudaSuccess) {   // give cached blocks back to the driver and retry once
            cudaGetLastError();
            trim(dev);
            e = cudaMalloc(out, bytes);
        }
        if (e == cudaSuccess) { std::lock_guard<std::mutex> g(mu); live[*out] = {bytes, dev}; }
        return e;
    }
    void release(void* p) {
        if (!p) return;
        std::lock_guard<std::mutex> g(mu);
        auto it = live.find(p);
        if (it == live.end()) { cudaFree(p); return; }
        free_list.push_back({p, it->second.first, it->second.second});
        live.erase(it);
    }
    void trim(int dev) {
        std::lock_guard<std::mutex> g(mu);
        for (const Blk& b : free_list) if (b.dev == dev) cudaFree(b.p);
        free_list.erase(std::remove_if(free_list.begin(), free_list.end(), [&](const Blk& b) { return b.dev == dev; }), free_list.end());
    }
};
static DevCache g_dev_cache;

template <class T>
struct DevArr {   // growable device array (never shrinks); returned to the cache with the owner
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap && p) return cudaSuccess;
        if (p) g_dev_cache.release(p);
        p = nullptr; cap = 0;
        void* q = nullptr;
        cudaError_t e = g_dev_cache.alloc(&q, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) { p = (T*)q; cap = std::max<size_t>(n, 1); }
        return e;
    }
    // room for n elements and their copy from the host queued on s; nothing at all (no allocation either) for n == 0
    cudaError_t upload(const T* h, size_t n, cudaStream_t s) {
        if (!n) return cudaSuccess;
        const cudaError_t e = reserve(n);
        return e == cudaSuccess ? cudaMemcpyAsync(p, h, n * sizeof(T), cudaMemcpyHostToDevice, s) : e;
    }
    cudaError_t upload(const std::vector<T>& h, cudaStream_t s) { return upload(h.data(), h.size(), s); }
    void release() { if (p) g_dev_cache.release(p); p = nullptr; cap = 0; }
    ~DevArr() { release(); }
    DevArr() = default;
    DevArr(const DevArr&) = delete;
    DevArr& operator=(const DevArr&) = delete;
};

static inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// A table-driven block-cipher kernel and the dynamic shared memory it is opted in to (ctx_create_single, enc::init_attributes;
// a kernel without any keeps the default) and launched with.  AES: Te0 or Td0 replicated per lane (32 KB), plus the inverse
// S-box (256 bytes) where the kernel may decrypt; Camellia: sp_hi | sp_lo (16 KB).
template <class F>
struct CipherKernel {
    F fn;
    int smem;
    bool opt_in() const { return !smem || cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess; }
};
constexpr int AES_SMEM = 256 * 32 * 4, AES_DEC_SMEM = AES_SMEM + 256, CAM_SMEM = 2 * 2048 * 4;
// decode cipher-tile slots (variant_of), in launch order; AES-CTR runs aes_ctr_tiles_kernel
static const CipherKernel<decltype(&decrypt_tiles_kernel<0, 1>)> DECRYPT_TILES[4] = {
    {decrypt_tiles_kernel<0, 1>, 0},              // gather of plain multi-body streams
    {decrypt_tiles_kernel<1, 0>, AES_DEC_SMEM},   // AES-CBC
    {decrypt_tiles_kernel<2, 1>, CAM_SMEM},       // Camellia-CTR
    {decrypt_tiles_kernel<2, 0>, CAM_SMEM}};      // Camellia-CBC
constexpr int ECB_SMEM = AES_DEC_SMEM;

// Expanded key schedule of one (cipher, key): encryption 1 AES-256, 2 Camellia-256
static DevKeys expand_key(const pna_ctx* ctx, uint8_t encryption, const uint8_t key[32]) {
    DevKeys dk;
    memset(&dk, 0, sizeof dk);
    if (encryption == 1) {
        AesKey ak; aes256_expand_key(&ctx->h_aes, key, &ak);
        memcpy(dk.aes_rk, ak.rk, sizeof ak.rk); memcpy(dk.aes_dk, ak.dk, sizeof ak.dk);
    } else {
        CamelliaKey ck; camellia256_expand_key(&ctx->h_cam, key, &ck);
        memcpy(dk.cam_ek, ck.ek, sizeof ck.ek); memcpy(dk.cam_dk, ck.dk, sizeof ck.dk);
    }
    return dk;
}
// The key schedules of one plan, one per distinct (cipher, key); entries refer to them by index
struct KeyTable {
    std::vector<DevKeys> keys;
    std::map<std::array<uint8_t, 33>, int> ids;
    int index(const pna_ctx* ctx, uint8_t encryption, const uint8_t key[32]) {
        std::array<uint8_t, 33> k;
        k[0] = encryption;
        memcpy(k.data() + 1, key, 32);
        auto it = ids.find(k);
        if (it == ids.end()) {
            it = ids.emplace(k, (int)keys.size()).first;
            keys.push_back(expand_key(ctx, encryption, key));
        }
        return it->second;
    }
};

// The reference's dispatch on an entry's compression, encryption and cipher mode (entry/read.rs:59-190): ST_UNSUPPORTED
// for a value it does not know, else ST_OK.  Decode and encode accept the same set.
static int32_t entry_mode_status(uint8_t compression, uint8_t encryption, uint8_t cipher_mode) {
    if (compression != PNA_COMPRESSION_NO && compression != PNA_COMPRESSION_DEFLATE && compression != PNA_COMPRESSION_ZSTD &&
        compression != PNA_COMPRESSION_XZ)
        return ST_UNSUPPORTED;
    if (encryption != PNA_ENCRYPTION_NO && encryption != PNA_ENCRYPTION_AES && encryption != PNA_ENCRYPTION_CAMELLIA)
        return ST_UNSUPPORTED;
    if (encryption != 0 && cipher_mode != PNA_CIPHER_CBC && cipher_mode != PNA_CIPHER_CTR && cipher_mode != PNA_CIPHER_GCM)
        return ST_UNSUPPORTED;
    return ST_OK;
}

// ------------------------------------------------------------------------------------------------
// Host span -> device image staging with range coalescing: spans that lie close together in host
// memory (e.g. the FDAT bodies of one mmap'd archive) travel in one cudaMemcpyAsync.
struct Stager {
    struct Range { const uint8_t* host; uint64_t len; uint64_t dev_off; };
    std::vector<Range> ranges;
    uint64_t total = 0;
    static constexpr uint64_t GAP = 64 * 1024;
    // Gaps between spans are carried along only inside a host range the caller DECLARED as one allocation (the archive
    // image of pna_cuda_decode_plan_create_in_image): bytes between independent allocations are not the caller's to read.
    const uint8_t* image = nullptr;
    uint64_t image_len = 0;
    bool inside(const uint8_t* p, uint64_t len) const { return image && p >= image && len <= image_len && (uint64_t)(p - image) <= image_len - len; }
    bool sealed = false;   // after the CRC spans were registered: later spans first try to resolve inside a range
    // returns the device offset of the span
    uint64_t add(const uint8_t* p, uint64_t len) {
        if (len == 0) return total;
        if (sealed) {   // ranges are sorted by host address (spans were registered in ascending order)
            size_t lo = 0, hi = ranges.size();
            while (lo < hi) { size_t mid = (lo + hi) / 2; if (ranges[mid].host <= p) lo = mid + 1; else hi = mid; }
            if (lo > 0) {
                const Range& r = ranges[lo - 1];
                if (p >= r.host && p + len <= r.host + r.len) return r.dev_off + (uint64_t)(p - r.host);
            }
            sealed = false;   // not covered (bodies without CRC spans): fall back to appending
            uint64_t off = add(p, len);
            sealed = true;
            return off;
        }
        if (!ranges.empty()) {
            Range& r = ranges.back();
            const uint8_t* end = r.host + r.len;
            const bool bridge = inside(r.host, r.len) && inside(p, len);
            if (p >= r.host && p <= end + (bridge ? GAP : 0)) {
                uint64_t off = r.dev_off + (uint64_t)(p - r.host);
                if (p + len > end) { r.len = (uint64_t)(p + len - r.host); total = r.dev_off + r.len; }
                return off;
            }
        }
        uint64_t dev = align_up(total, 256) + ((uintptr_t)p & 15);   // keep the host pointer's 16-byte phase
        ranges.push_back({p, len, dev});
        total = dev + len;
        return dev;
    }
    int upload(pna_ctx* ctx, uint8_t* d_base) {
        for (const Range& r : ranges) CK(cudaMemcpyAsync(d_base + r.dev_off, r.host, r.len, cudaMemcpyHostToDevice, ctx->stream));
        return PNA_OK;
    }
};

constexpr int PNA_N_STAGES = 9;
static const char* const PNA_STAGE_NAMES[PNA_N_STAGES] = {"crc", "cipher", "zstd_scan", "zstd_seq", "zstd_lit", "zstd_prefix", "zstd_lz", "inflate", "store"};

// GCM STREAM (cipher mode 2) tables of a plan on the device: segments, 16 KiB warp tiles (the first n_tiles_aes of them AES,
// the rest Camellia) with a partial GHASH each, and one key reference and power table per entry
struct GcmDev {
    DevArr<gcm::GcmSeg> segs;
    DevArr<gcm::GcmTile> tiles;
    DevArr<gcm::GcmKeyRef> refs;
    DevArr<gcm::GcmPow> pows;
    DevArr<gcm::G128> partial;
    uint32_t n_segs = 0, n_tiles = 0, n_tiles_aes = 0, n_keys = 0;
};

// chunk-CRC spans a decode plan verifies on its uploaded image (pna_cuda_decode_plan_create_crc / _in_image)
struct CrcReq { const pna_span* spans; const uint32_t* expect; const int32_t* entry_of; uint32_t n; const uint8_t* image; uint64_t image_len; };

namespace pna { namespace multi { struct Plan; } }
// ------------------------------------------------------------------------------------------------
struct pna_plan {
    pna::multi::Plan* multi = nullptr;   // set: a plan of a multi-device context (multi_host.cuh); everything below is unused then
    pna_ctx* ctx = nullptr;
    int kind = 0;   // 0 decode, 1 encode
    uint32_t n = 0;
    bool prepared = false, need_sizing = false;
    uint64_t stream_bytes = 0, plain_bytes = 0, launches_per_run = 0;
    // host metadata
    std::vector<EntryRec> h_entries;
    std::vector<Segment> h_segs;
    KeyTable h_keys;
    std::vector<CipherTile> h_tiles[4];   // by variant_of: 0 gather, 1 aes-cbc, 2 camellia-ctr, 3 camellia-cbc
    std::vector<CtrTile> h_ctr_tiles;     // aes-ctr
    std::vector<uint32_t> h_store, h_deflate, h_xz;
    // GCM STREAM (cipher mode 2): the host side of `gcm`
    std::vector<gcm::GcmSeg> h_gcm_segs;
    std::vector<gcm::GcmTile> h_gcm_tiles;
    std::vector<gcm::GcmKeyRef> h_gcm_refs;
    GcmDev gcm;
    std::vector<inf::InfStream> h_inf;          // deflate streams of the two-stage path (tokens -> LZ -> Adler)
    std::vector<uint32_t> h_deflate_big;        // streams of 2 GiB and more: one-thread-per-stream kernel
    std::vector<zs::ZEntry> h_ze;
    std::vector<CopyJob> h_copy;
    uint64_t image_bytes = 0, buf_bytes = 0, out_bytes = 0;
    // device
    DevArr<uint8_t> d_buf, d_out, d_lits;
    DevArr<EntryRec> d_entries, d_entries_init;
    DevArr<Segment> d_segs;
    DevArr<DevKeys> d_keys;
    DevArr<CipherTile> d_tiles[4];
    DevArr<CtrTile> d_ctr_tiles;
    DevArr<uint32_t> d_deflate, d_seq_order, d_lit_order, d_counts, d_lz_order;
    DevArr<zs::SeqRec> d_seqs;
    DevArr<zs::ZEntry> d_ze;
    DevArr<zs::LzUnit> d_lz_units;   // one per frame
    uint32_t n_lz_units = 0;
    uint64_t lz_avg_unit_comp = 0;   // compressed bytes per unit, for the choice of the LZ kernel variant
    DevArr<zs::ZBlock> d_blocks;
    DevArr<zs::WalkRec> d_walk;        // block headers as the (serial) frame walk found them
    // entries decoded block-parallel inside their frames (kernels_zstd_pj.cuh): segments, pointer scratch, round flags
    std::vector<zs::PjSeg> h_pj_segs;
    DevArr<zs::PjSeg> d_pj_segs;
    DevArr<int32_t> d_pj_ptr;
    DevArr<uint2> d_pj_cpos;
    DevArr<uint32_t> d_pj_flags;
    DevArr<uint8_t> d_pj_tiles;        // one byte per 1024 pointers, two copies (ping-pong between rounds)
    uint64_t pj_tile_stride = 0;
    uint32_t pj_max_blocks = 0;
    DevArr<uint64_t> d_lit_base, d_seq_base;
    DevArr<inf::InfStream> d_inf;
    DevArr<uint32_t> d_xz;
    // chunk-parallel xz (kernels_xz.cuh): windows of the streams' outputs, built with the output layout
    std::vector<uint2> h_xz_map;
    std::vector<uint32_t> h_xz_win_begin;
    DevArr<uint2> d_xz_map;
    DevArr<uint32_t> d_xz_win_begin;
    DevArr<xz::XzWin> d_xz_wins;
    DevArr<uint8_t> d_inf_lits;
    DevArr<zs::SeqRec> d_inf_recs;
    DevArr<zs::ZBlock> d_inf_blocks;
    DevArr<zs::ZEntry> d_inf_ze;
    DevArr<inf::InfTrailer> d_inf_tr;
    DevArr<CopyJob> d_copy;
    uint32_t n_blocks = 0;
    uint64_t lit_total = 0, seq_total = 0;
    std::vector<uint64_t> h_out_len;   // decoded length per entry (pna_cuda_decode_plan_lengths)
    // per-stage CUDA events of the last run (cipher, zstd scan, entropy, prefix, lz, inflate, store)
    cudaEvent_t ev[PNA_N_STAGES + 1] = {};
    bool ev_ready = false, ev_recorded = false;
    bool sized_entropy = false;   // prepare() already ran entropy+prefix / inflate sizing on the live table
    DevArr<uint64_t> d_layout;
    // optional chunk-CRC verification riding on the same uploaded image (seam 1 fused into the plan)
    std::vector<CrcTile> h_crc_tiles;
    std::vector<uint32_t> h_crc_first, h_crc_expect;
    std::vector<int32_t> h_crc_entry;
    DevArr<CrcTile> d_crc_tiles;
    DevArr<uint32_t> d_crc_first, d_crc_expect, d_crc_raw, d_crc_val, d_crc_broken;
    DevArr<int32_t> d_crc_entry;
    uint32_t n_crc = 0;
    // encode side
    enc::EncodePlan* enc = nullptr;
    ~pna_plan() {
        if (ev_ready) for (auto& e : ev) { if (ctx) ctx->ev_pool.push_back(e); else cudaEventDestroy(e); }
        if (enc) enc::destroy(enc);
    }
};

#include "multi_host.cuh"

// ------------------------------------------------------------------------------------------------
extern "C" const char* pna_cuda_strerror(int32_t s) {
    switch (s) {
        case PNA_OK: return "ok";
        case PNA_E_INVALID_DATA: return "invalid data";
        case PNA_E_UNEXPECTED_EOF: return "unexpected end of stream";
        case PNA_E_INVALID_INPUT: return "invalid input";
        case PNA_E_UNSUPPORTED: return "unsupported";
        case PNA_E_NOSPACE: return "output buffer too small";
        case PNA_E_OOM: return "out of memory";
        case PNA_E_INTERNAL: return "internal error";
        case PNA_E_CUDA: return "CUDA failure";
        case PNA_E_BAD_ARG: return "bad argument";
        default: return "unknown";
    }
}

static int ctx_create_single(pna_ctx** out, int device_id);
extern "C" int pna_cuda_init(pna_ctx** out, const int* device_ids, int n_devices) {
    if (!out || n_devices < 0) return PNA_E_BAD_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return PNA_E_CUDA;   // no fallback: fail loudly
    std::vector<int> ids;
    if (device_ids) ids.assign(device_ids, device_ids + n_devices);
    else for (int d = 0; d < (n_devices ? n_devices : count); d++) ids.push_back(d);   // NULL: the first n (0: all visible) devices
    if (ids.empty()) return PNA_E_BAD_ARG;
    for (size_t i = 0; i < ids.size(); i++) {
        if (ids[i] < 0 || ids[i] >= count) return PNA_E_BAD_ARG;
        for (size_t j = 0; j < i; j++) if (ids[j] == ids[i]) return PNA_E_BAD_ARG;
    }
    if (ids.size() == 1) return ctx_create_single(out, ids[0]);
    pna_ctx* root = new pna_ctx();
    root->device = ids[0];
    for (int d : ids) {
        pna_ctx* c = nullptr;
        const int rc = ctx_create_single(&c, d);
        if (rc != PNA_OK) { for (pna_ctx* q : root->devs) pna_cuda_destroy(q); delete root; return rc; }
        root->devs.push_back(c);
    }
    root->sm_count = root->devs[0]->sm_count;
    *out = root;
    return PNA_OK;
}
static int ctx_create_single(pna_ctx** out, int device_id) {
    pna_ctx* ctx = new pna_ctx();
    ctx->device = device_id;
    if (cudaSetDevice(device_id) != cudaSuccess) { delete ctx; return PNA_E_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_id) != cudaSuccess || prop.major < 10) { delete ctx; return PNA_E_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return PNA_E_CUDA; }
    if (cudaEventCreateWithFlags(&ctx->sync_ev, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return PNA_E_CUDA; }
    CrcConsts* hc = new CrcConsts();
    crc_make_consts(hc);
    aes_make_tables(&ctx->h_aes);
    camellia_make_tables(&ctx->h_cam);
    bool ok = cudaMalloc(&ctx->d_crc, sizeof(CrcConsts)) == cudaSuccess &&
              cudaMalloc(&ctx->d_aes, sizeof(AesTables)) == cudaSuccess &&
              cudaMalloc(&ctx->d_cam, sizeof(CamelliaTables)) == cudaSuccess &&
              cudaMemcpy(ctx->d_crc, hc, sizeof(CrcConsts), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_aes, &ctx->h_aes, sizeof(AesTables), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_cam, &ctx->h_cam, sizeof(CamelliaTables), cudaMemcpyHostToDevice) == cudaSuccess;
    delete hc;
    // opt in to the large dynamic shared memory the table-driven kernels use
    ok = ok && cudaFuncSetAttribute(aes_ctr_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AES_CTR_TILES_SMEM) == cudaSuccess;
    for (const auto& k : DECRYPT_TILES) ok = ok && k.opt_in();
    ok = ok && cudaFuncSetAttribute(ecb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ECB_SMEM) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(gcm::gcm_tiles_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, gcm::gcm_tiles_smem<1>()) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(gcm::gcm_tiles_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, gcm::gcm_tiles_smem<2>()) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(gcm::gcm_tiles_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, gcm::gcm_tiles_smem<1>()) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(gcm::gcm_tiles_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, gcm::gcm_tiles_smem<2>()) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(inf::inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(sizeof(inf::Tables) * inf::INFLATE_CTA)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(crc_tiles_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CRC_WIDE_SMEM) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(xz::xz_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xz::XZ_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(xz::xz_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xz::XZ_WIN_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(inf::inflate_tokens_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)inf::TOKEN_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(zs::zstd_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zs::SEQ_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(zs::zstd_lit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zs::LIT_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(zs::zstd_lz_kernel<zs::LzSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zs::LzSmall::BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(zs::zstd_lz_kernel<zs::LzBig>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zs::LzBig::BYTES) == cudaSuccess;
    ok = ok && enc::init_attributes();
    if (!ok) { pna_cuda_destroy(ctx); return PNA_E_CUDA; }
    *out = ctx;
    return PNA_OK;
}

extern "C" void pna_cuda_destroy(pna_ctx* ctx) {
    if (!ctx) return;
    if (!ctx->devs.empty()) { for (pna_ctx* c : ctx->devs) pna_cuda_destroy(c); delete ctx; return; }
    cudaSetDevice(ctx->device);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
    if (ctx->sync_ev) cudaEventDestroy(ctx->sync_ev);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    g_dev_cache.trim(ctx->device);
    if (ctx->d_crc) cudaFree(ctx->d_crc);
    if (ctx->d_aes) cudaFree(ctx->d_aes);
    if (ctx->d_cam) cudaFree(ctx->d_cam);
    delete ctx;
}
extern "C" const char* pna_cuda_last_error(pna_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }
extern "C" void* pna_cuda_host_alloc(pna_ctx* ctx, uint64_t bytes) {
    if (!ctx) return nullptr;
    cudaSetDevice(ctx->device);
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;   // pinned for every device of the process
    return p;
}
extern "C" void pna_cuda_host_free(pna_ctx* ctx, void* p) { if (p) cudaFreeHost(p); }
extern "C" int pna_cuda_device_count(pna_ctx* ctx) { return !ctx ? 0 : ctx->devs.empty() ? 1 : (int)ctx->devs.size(); }
extern "C" int pna_cuda_device_id(pna_ctx* ctx, int i) {
    if (!ctx || i < 0 || i >= pna_cuda_device_count(ctx)) return -1;
    return ctx->devs.empty() ? ctx->device : ctx->devs[i]->device;
}
extern "C" void* pna_cuda_stream(pna_ctx* ctx) { return !ctx ? nullptr : ctx->devs.empty() ? (void*)ctx->stream : (void*)ctx->devs[0]->stream; }
extern "C" uint64_t pna_cuda_launch_count(pna_ctx* ctx) {
    if (!ctx) return 0;
    uint64_t n = ctx->launches;
    for (pna_ctx* c : ctx->devs) n += c->launches;
    return n;
}

// Transfer yardstick for end-to-end numbers: the same pinned <-> HBM copies a step makes, timed with CUDA events -- H2D
// alone, D2H alone, and both directions at once on two streams (what the pipelined host layer does; PCIe is full duplex but
// the directions are not independent).  Run by every rank at the same time it gives the box's concurrent transfer floor.
extern "C" int pna_cuda_transfer_probe(pna_ctx* ctx, const uint8_t* h2d_src, uint64_t h2d_bytes, uint8_t* d2h_dst, uint64_t d2h_bytes,
                                       float* h2d_ms, float* d2h_ms, float* both_ms) {
    if (!ctx || (!h2d_src && h2d_bytes) || (!d2h_dst && d2h_bytes)) return PNA_E_BAD_ARG;
    if (!ctx->devs.empty()) ctx = ctx->devs[0];
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    DevArr<uint8_t> d_in, d_out;
    CK(d_in.reserve(h2d_bytes + 256)); CK(d_out.reserve(d2h_bytes + 256));
    cudaStream_t s2 = nullptr;
    cudaEvent_t e[4] = {};
    CK(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
    for (auto& x : e) CK(cudaEventCreate(&x));
    int rc = PNA_OK;
    auto ck2 = [&](cudaError_t err) { if (err != cudaSuccess && rc == PNA_OK) { ctx->fail("transfer probe", err); rc = PNA_E_CUDA; } };
    float t = 0;
    // warm-up (page tables of the pinned ranges, first-touch of the device arenas)
    if (h2d_bytes) ck2(cudaMemcpyAsync(d_in.p, h2d_src, h2d_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (d2h_bytes) ck2(cudaMemcpyAsync(d2h_dst, d_out.p, d2h_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ck2(ctx->sync());
    ck2(cudaEventRecord(e[0], ctx->stream));
    if (h2d_bytes) ck2(cudaMemcpyAsync(d_in.p, h2d_src, h2d_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ck2(cudaEventRecord(e[1], ctx->stream));
    if (d2h_bytes) ck2(cudaMemcpyAsync(d2h_dst, d_out.p, d2h_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ck2(cudaEventRecord(e[2], ctx->stream));
    ck2(ctx->sync());
    if (rc == PNA_OK) { cudaEventElapsedTime(&t, e[0], e[1]); if (h2d_ms) *h2d_ms = t; cudaEventElapsedTime(&t, e[1], e[2]); if (d2h_ms) *d2h_ms = t; }
    // both directions at once: s2 starts behind the common start event
    ck2(cudaEventRecord(e[0], ctx->stream));
    ck2(cudaStreamWaitEvent(s2, e[0], 0));
    if (h2d_bytes) ck2(cudaMemcpyAsync(d_in.p, h2d_src, h2d_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (d2h_bytes) ck2(cudaMemcpyAsync(d2h_dst, d_out.p, d2h_bytes, cudaMemcpyDeviceToHost, s2));
    ck2(cudaEventRecord(e[3], s2));
    ck2(cudaStreamWaitEvent(ctx->stream, e[3], 0));
    ck2(cudaEventRecord(e[1], ctx->stream));
    ck2(ctx->sync());
    if (rc == PNA_OK) { cudaEventElapsedTime(&t, e[0], e[1]); if (both_ms) *both_ms = t; }
    for (auto& x : e) cudaEventDestroy(x);
    cudaStreamDestroy(s2);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// seam 1: CRC
// CRC-32 of n spans of img, each cut into CRC_TILE tiles (first[i]: the first tile of span i): raw CRCs of the tiles, then
// one fold per span, which starts from `init` (the register after a prefix the CRC covers but the image does not hold)
static int launch_chunk_crc(pna_ctx* ctx, const uint8_t* img, const CrcTile* tiles, uint32_t nt, uint32_t* raw, const uint32_t* first,
                            uint32_t n, uint32_t* crc, uint32_t init = 0xFFFFFFFFu) {
    launch_crc_tiles(ctx->stream, ctx->sm_count, img, tiles, nt, ctx->d_crc, raw);
    LAUNCHED();
    crc_combine_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(tiles, raw, first, n, nt, ctx->d_crc, crc, init);
    LAUNCHED();
    return PNA_OK;
}
// the next span (l bytes at device offset o): its first tile into `first`, its CRC_TILE tiles (one, empty, for l == 0) into `tiles`
static void add_crc_span(std::vector<CrcTile>& tiles, std::vector<uint32_t>& first, uint64_t o, uint64_t l) {
    const uint32_t i = (uint32_t)first.size();
    first.push_back((uint32_t)tiles.size());
    do {
        uint32_t t = (uint32_t)std::min<uint64_t>(l, CRC_TILE);
        tiles.push_back({o, t, i});
        o += t; l -= t;
    } while (l);
}
static int crc_run(pna_ctx* ctx, const uint8_t* d_img, const std::vector<uint64_t>& off, const uint64_t* len, uint32_t n,
                   uint32_t* crc_out) {
    std::vector<CrcTile> tiles;
    std::vector<uint32_t> first;
    tiles.reserve(n); first.reserve(n);
    for (uint32_t i = 0; i < n; i++) add_crc_span(tiles, first, off[i], len[i]);
    const uint32_t nt = (uint32_t)tiles.size();
    DevArr<CrcTile> d_tiles; DevArr<uint32_t> d_first, d_raw, d_crc;
    CK(d_tiles.upload(tiles, ctx->stream)); CK(d_first.upload(first, ctx->stream));
    CK(d_raw.reserve(nt)); CK(d_crc.reserve(n));
    const int rc = launch_chunk_crc(ctx, d_img, d_tiles.p, nt, d_raw.p, d_first.p, n, d_crc.p);
    if (rc) return rc;
    CK(cudaMemcpyAsync(crc_out, d_crc.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    return PNA_OK;
}

extern "C" int pna_cuda_crc32(pna_ctx* ctx, const pna_span* spans, uint32_t n, uint32_t* crc_out) {
    if (!ctx || (!spans && n) || (!crc_out && n)) return PNA_E_BAD_ARG;
    if (n == 0) return PNA_OK;
    if (!ctx->devs.empty()) return multi::crc32(ctx, spans, n, crc_out);
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    Stager st;
    std::vector<uint64_t> off(n), len(n);
    for (uint32_t i = 0; i < n; i++) { off[i] = st.add(spans[i].ptr, spans[i].len); len[i] = spans[i].len; }
    DevArr<uint8_t> d_img;
    CK(d_img.reserve(st.total + 64));
    int rc = st.upload(ctx, d_img.p);
    if (rc == PNA_OK) rc = crc_run(ctx, d_img.p, off, len.data(), n, crc_out);
    ctx->sync();
    return rc;
}

extern "C" int pna_cuda_crc32_image(pna_ctx* ctx, const uint8_t* image, uint64_t image_len, const uint64_t* span_off,
                                    const uint64_t* span_len, uint32_t n, uint32_t* crc_out) {
    if (!ctx || (!image && image_len) || ((!span_off || !span_len || !crc_out) && n)) return PNA_E_BAD_ARG;
    if (n == 0) return PNA_OK;
    for (uint32_t i = 0; i < n; i++)
        if (span_off[i] > image_len || span_len[i] > image_len - span_off[i]) return PNA_E_BAD_ARG;
    if (!ctx->devs.empty()) return multi::crc32_image(ctx, image, span_off, span_len, n, crc_out);
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    DevArr<uint8_t> d_img;
    CK(d_img.reserve(image_len + 64));
    cudaError_t e = cudaMemcpyAsync(d_img.p, image, image_len, cudaMemcpyHostToDevice, ctx->stream);
    int rc = PNA_OK;
    if (e != cudaSuccess) { ctx->fail("image upload", e); rc = PNA_E_CUDA; }
    std::vector<uint64_t> off(span_off, span_off + n);
    if (rc == PNA_OK) rc = crc_run(ctx, d_img.p, off, span_len, n, crc_out);
    ctx->sync();
    return rc;
}

// ------------------------------------------------------------------------------------------------
// seam 2: decode
// cipher-tile slot (DECRYPT_TILES) of an entry that is neither AES-CTR nor GCM
static int variant_of(const EntryRec& e) {
    if (e.encryption == 0) return 0;
    return e.encryption == PNA_ENCRYPTION_AES ? 1 : e.cipher_mode == PNA_CIPHER_CTR ? 2 : 3;
}

// Upper bound of what a compressed stream of `comp_len` bytes can decode to: zstd emits at most one 128 KiB block per 4
// stream bytes (RLE block: 3-byte header + 1 byte), deflate at most 1032 bytes per stream byte, store is the identity.
static uint64_t decode_size_bound(uint8_t compression, uint64_t comp_len) {
    if (compression == PNA_COMPRESSION_ZSTD) return comp_len > ((uint64_t)1 << 44) ? UINT64_MAX / 2 : (comp_len / 3 + 2) * 131072ull;
    if (compression == PNA_COMPRESSION_DEFLATE) return comp_len > ((uint64_t)1 << 50) ? UINT64_MAX / 2 : comp_len * 1032ull + 1024;
    if (compression == PNA_COMPRESSION_XZ) return comp_len > ((uint64_t)1 << 40) ? UINT64_MAX / 2 : (comp_len / 6 + 1) * (2ull << 20);   // LZMA2 chunk: <= 2 MiB from >= 6 bytes
    return comp_len;
}
extern "C" uint64_t pna_cuda_decode_size_bound(uint8_t compression, uint64_t stream_len) { return decode_size_bound(compression, stream_len); }
// whether a size hint (fSIZ) is used to lay out the output, or ignored in favour of the exact sizing pass
static bool size_hint_trusted(uint8_t compression, uint64_t comp_len, uint64_t hint) {
    if (hint == UINT64_MAX || hint > decode_size_bound(compression, comp_len)) return false;
    return !(hint > ((uint64_t)1 << 30) && hint / 256 > comp_len);   // huge both absolutely and relative to the stream
}
extern "C" int pna_cuda_size_hint_trusted(uint8_t compression, uint64_t stream_len, uint64_t hint) { return size_hint_trusted(compression, stream_len, hint) ? 1 : 0; }
// AES-CTR tiles of entry i (aes_ctr_tiles_kernel): cut at body boundaries and after CTR_TILE_RUNS counter runs; a block that
// straddles two bodies becomes a one-block tile gathered through the segments.  The IV is read here, from the host bodies.
static void ctr_tiles(pna_plan* P, const pna_decode_desc& d, uint32_t i) {
    const EntryRec& e = P->h_entries[i];
    uint8_t ivb[16];
    uint64_t got = 0;
    for (uint32_t b = 0; b < d.n_bodies && got < 16; b++) {
        const uint64_t k = std::min<uint64_t>(d.bodies[b].len, 16 - got);
        if (k) memcpy(ivb + got, d.bodies[b].ptr, k);
        got += k;
    }
    uint32_t iv[4];
    memcpy(iv, ivb, 16);
    const Segment* sg = P->h_segs.data() + e.seg_begin;
    const uint64_t clen = e.comp_len, nb = (clen + 15) / 16;
    uint32_t si = 0;
    for (uint64_t b = 0; b < nb;) {
        const uint64_t pos = 16 + 16 * b, rest = clen - 16 * b;
        while (si + 1 < e.n_segs && sg[si + 1].pos <= pos) si++;
        const uint64_t seg_end = si + 1 < e.n_segs ? sg[si + 1].pos : e.stream_len;
        CtrTile t;
        memset(&t, 0, sizeof t);
        ctr128be_add(iv, b, t.ctr);
        t.dst = e.comp_off + 16 * b;
        t.key_idx = (uint32_t)e.key_idx;
        t.entry = i;
        t.pos = pos;
        uint64_t n;
        if (std::min<uint64_t>(rest, 16) > seg_end - pos) {   // straddles two bodies
            t.src = CTR_TILE_SLOW;
            n = 1;
        } else {
            t.src = sg[si].img_off + (pos - sg[si].pos);
            n = rest <= seg_end - pos ? nb - b : (seg_end - pos) / 16;
            n = std::min<uint64_t>(n, 256 * CTR_TILE_RUNS - (t.ctr[3] >> 24));
        }
        t.n_bytes = (uint32_t)std::min<uint64_t>(16 * n, rest);
        P->h_ctr_tiles.push_back(t);
        b += n;
    }
}

static int decode_plan_build(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, const uint64_t* caps, const CrcReq* crc,
                             pna_plan* P) {
    P->ctx = ctx; P->kind = 0; P->n = n;
    P->h_entries.resize(n);
    Stager st;
    if (crc) { st.image = crc->image; st.image_len = crc->image_len; }
    // chunk spans (type||data) first: they start 4 bytes before the bodies, so bodies fall into the same ranges
    // when both are registered in address order; spans and bodies may also interleave arbitrarily.
    std::vector<uint64_t> crc_off;
    if (crc && crc->n && !crc->spans) return PNA_E_BAD_ARG;
    if (crc && crc->n) {
        // merge-register spans and bodies in ascending host address order so that ranges coalesce
        P->n_crc = crc->n;
        crc_off.resize(crc->n);
        std::vector<uint32_t> order(crc->n);
        for (uint32_t i = 0; i < crc->n; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return crc->spans[a].ptr < crc->spans[b].ptr; });
        for (uint32_t k : order) {
            if (crc->spans[k].len && !crc->spans[k].ptr) return PNA_E_BAD_ARG;
            crc_off[k] = st.add(crc->spans[k].ptr, crc->spans[k].len);
        }
        st.sealed = true;   // bodies now only look up / extend; see Stager::add
    }
    uint64_t comp_extra = 0;   // bytes needed in the comp region (decrypted / gathered streams)
    std::vector<uint8_t> needs_copy(n, 0);
    std::vector<gcm::GcmSeg> gcm_walk;            // segments in entry order
    std::map<uint32_t, uint64_t> gcm_len;         // entry -> ciphertext bytes without header and tags
    for (uint32_t i = 0; i < n; i++) {
        const pna_decode_desc& d = descs[i];
        EntryRec& e = P->h_entries[i];
        memset(&e, 0, sizeof e);
        e.compression = d.compression; e.encryption = d.encryption; e.cipher_mode = d.cipher_mode;
        e.seg_begin = P->h_segs.size();
        e.key_idx = -1;
        uint64_t pos = 0;
        for (uint32_t b = 0; b < d.n_bodies; b++) {
            if (d.bodies[b].len == 0) continue;
            if (!d.bodies[b].ptr) return PNA_E_BAD_ARG;
            P->h_segs.push_back({st.add(d.bodies[b].ptr, d.bodies[b].len), pos});
            pos += d.bodies[b].len;
        }
        e.n_segs = (uint32_t)(P->h_segs.size() - e.seg_begin);
        e.stream_len = pos;
        P->stream_bytes += pos;
        // host-side validation == the reference's dispatch (entry/read.rs:59-190)
        e.status = entry_mode_status(d.compression, d.encryption, d.cipher_mode);
        if (e.status != ST_OK) continue;
        if (d.encryption != 0 && d.cipher_mode == PNA_CIPHER_GCM) {
            // stream header + segment walk (entry/read.rs:105-118, aead.rs:134-148, gcm.rs:206-262); every layout violation
            // is an AeadError == InvalidData (error.rs:67-74)
            uint8_t hdr[gcm::GCM_HEADER_LEN];
            uint64_t got = 0;
            for (uint32_t b = 0; b < d.n_bodies && got < sizeof hdr; b++) {
                const uint64_t k = std::min<uint64_t>(d.bodies[b].len, sizeof hdr - got);
                if (k) memcpy(hdr + got, d.bodies[b].ptr, k);
                got += k;
            }
            const uint32_t seg = got == sizeof hdr ? ((uint32_t)hdr[39] << 24 | (uint32_t)hdr[40] << 16 | (uint32_t)hdr[41] << 8 | hdr[42]) : 0;
            if (got < sizeof hdr || seg == 0 || seg > gcm::GCM_MAX_SEGMENT) e.status = ST_INVALID_DATA;
            else {
                const size_t seg0 = gcm_walk.size();
                uint64_t rest = pos - sizeof hdr, at = sizeof hdr, plain = 0;
                for (uint64_t i = 0;; i++) {
                    const uint64_t take = std::min<uint64_t>(rest, (uint64_t)seg + gcm::GCM_TAG_LEN);
                    const bool is_final = take == rest;
                    if (take < gcm::GCM_TAG_LEN || i > 0xFFFFFFFFull) { e.status = ST_INVALID_DATA; break; }   // malformed / truncated
                    gcm::GcmSeg g;
                    memset(&g, 0, sizeof g);
                    uint8_t nonce[12];
                    memcpy(nonce, hdr + 32, 7);
                    nonce[7] = (uint8_t)(i >> 24); nonce[8] = (uint8_t)(i >> 16); nonce[9] = (uint8_t)(i >> 8); nonce[10] = (uint8_t)i;
                    nonce[11] = is_final ? 1 : 0;   // aead.rs:210-217
                    memcpy(g.nonce, nonce, 12);
                    g.entry = (uint32_t)(&e - P->h_entries.data());
                    g.ct_pos = at; g.ct_len = take - gcm::GCM_TAG_LEN; g.dst_off = plain;   // + comp_off once that is known
                    gcm_walk.push_back(g);
                    plain += g.ct_len; at += take; rest -= take;
                    if (is_final) break;
                }
                if (e.status != ST_OK) gcm_walk.resize(seg0);
                else gcm_len[(uint32_t)(&e - P->h_entries.data())] = plain;
            }
        }
        else if (d.encryption != 0 && pos < 16)
            e.status = ST_UNEXPECTED_EOF;   // read_exact(iv)
        else if (d.encryption != 0 && d.cipher_mode == PNA_CIPHER_CBC && ((pos - 16) < 16 || (pos - 16) % 16))
            e.status = ST_UNEXPECTED_EOF;   // cipher/block/read.rs:36,90
        if (e.status != ST_OK) continue;
        if (d.encryption) {
            e.key_idx = P->h_keys.index(ctx, d.encryption, d.key);
            e.comp_len = d.cipher_mode == PNA_CIPHER_GCM ? gcm_len[i] : pos - 16;   // CBC: rewritten by the kernel after unpadding
            needs_copy[i] = 1;
        } else {
            e.comp_len = pos;
            needs_copy[i] = e.n_segs > 1;
        }
        if (needs_copy[i]) comp_extra += align_up(e.comp_len, 16) + 16;
    }
    P->image_bytes = align_up(st.total, 256);
    if (P->n_crc) {
        P->h_crc_expect.assign(crc->expect, crc->expect + crc->n);
        P->h_crc_entry.assign(crc->entry_of, crc->entry_of + crc->n);
        for (uint32_t i = 0; i < P->n_crc; i++) add_crc_span(P->h_crc_tiles, P->h_crc_first, crc_off[i], crc->spans[i].len);
    }
    // comp region right behind the image
    uint64_t cur = P->image_bytes;
    for (uint32_t i = 0; i < n; i++) {
        EntryRec& e = P->h_entries[i];
        if (e.status != ST_OK) continue;
        if (needs_copy[i]) {
            e.comp_off = cur;
            cur += align_up(e.comp_len, 16) + 16;
            const uint64_t nb = (e.comp_len + 15) / 16;
            if (e.encryption && e.cipher_mode == PNA_CIPHER_GCM) continue;   // tiled per segment below
            if (e.encryption == PNA_ENCRYPTION_AES && e.cipher_mode == PNA_CIPHER_CTR) {
                ctr_tiles(P, descs[i], i);
                continue;
            }
            std::vector<CipherTile>& tv = P->h_tiles[variant_of(e)];
            for (uint64_t b0 = 0; b0 < nb; b0 += CIPHER_TILE_BLOCKS)
                tv.push_back({i, (uint32_t)std::min<uint64_t>(CIPHER_TILE_BLOCKS, nb - b0), b0});
        } else {
            e.comp_off = e.n_segs ? P->h_segs[e.seg_begin].img_off : 0;
        }
    }
    P->buf_bytes = cur + 256;
    if (!gcm_walk.empty()) {
        // AES segments first, then Camellia (one kernel each); the first tile of a segment is the short one
        std::map<uint32_t, uint32_t> pow_of;
        for (int pass = 1; pass <= 2; pass++) {
            for (const gcm::GcmSeg& w : gcm_walk) {
                if (P->h_entries[w.entry].encryption != pass) continue;
                gcm::GcmSeg g = w;
                const EntryRec& ge = P->h_entries[g.entry];
                auto it = pow_of.find(g.entry);
                if (it == pow_of.end()) {
                    it = pow_of.emplace(g.entry, (uint32_t)P->h_gcm_refs.size()).first;
                    P->h_gcm_refs.push_back({ge.key_idx, (uint32_t)ge.encryption});
                }
                g.pow_idx = it->second;
                g.key_idx = ge.key_idx; g.enc = ge.encryption;
                g.src_seg_begin = ge.seg_begin; g.src_n_segs = ge.n_segs; g.src_len = ge.stream_len;
                g.dst_off += ge.comp_off;
                const uint64_t nb = (g.ct_len + 15) / 16;
                g.first_tile = (uint32_t)P->h_gcm_tiles.size();
                const uint32_t sidx = (uint32_t)P->h_gcm_segs.size();
                uint64_t b0 = 0;
                const uint64_t head = nb % gcm::GCM_TILE_BLOCKS;
                if (head) { P->h_gcm_tiles.push_back({sidx, (uint32_t)head, 0}); b0 = head; }
                for (; b0 < nb; b0 += gcm::GCM_TILE_BLOCKS) P->h_gcm_tiles.push_back({sidx, gcm::GCM_TILE_BLOCKS, b0});
                g.n_tiles = (uint32_t)P->h_gcm_tiles.size() - g.first_tile;
                P->h_gcm_segs.push_back(g);
            }
            if (pass == 1) P->gcm.n_tiles_aes = (uint32_t)P->h_gcm_tiles.size();
        }
    }
    // decode lists
    bool all_caps = true;
    for (uint32_t i = 0; i < n; i++) {
        EntryRec& e = P->h_entries[i];
        uint64_t cap = caps ? caps[i] : descs[i].raw_size_hint;
        // fSIZ is untrusted input (the reference never sizes anything from it: its readers are stream-driven).  No stream of
        // comp_len bytes can decode to more than `bound`, so a larger capacity is clamped (a caller's buffer) or, for a mere
        // hint, ignored in favour of the exact sizing pass; so is a hint that is huge both absolutely and relative to the stream.
        const uint64_t bound = decode_size_bound(e.compression, e.comp_len);
        if (caps) { if (cap != UINT64_MAX && cap > bound) cap = bound; }
        else if (!size_hint_trusted(e.compression, e.comp_len, cap)) cap = UINT64_MAX;
        e.out_cap = cap;
        if (e.status != ST_OK) { e.out_cap = 0; continue; }
        if (cap == UINT64_MAX) all_caps = false;
        if (e.compression == PNA_COMPRESSION_NO) P->h_store.push_back(i);
        else if (e.compression == PNA_COMPRESSION_DEFLATE) P->h_deflate.push_back(i);
        else if (e.compression == PNA_COMPRESSION_XZ) P->h_xz.push_back(i);
        else { zs::ZEntry z; memset(&z, 0, sizeof z); z.entry = i; P->h_ze.push_back(z); }
    }
    P->need_sizing = !all_caps;
    std::stable_sort(P->h_deflate.begin(), P->h_deflate.end(), [&](uint32_t a, uint32_t b) { return P->h_entries[a].comp_len > P->h_entries[b].comp_len; });
    std::stable_sort(P->h_xz.begin(), P->h_xz.end(), [&](uint32_t a, uint32_t b) { return P->h_entries[a].comp_len > P->h_entries[b].comp_len; });
    // device arrays + upload; entries, segments and keys get room even when there are none: kernels take their pointers
    CK(P->d_buf.reserve(P->buf_bytes));
    CK(P->d_entries.reserve(n)); CK(P->d_entries_init.reserve(n));
    CK(P->d_segs.reserve(P->h_segs.size()));
    CK(P->d_keys.reserve(P->h_keys.keys.size()));
    int rc = st.upload(ctx, P->d_buf.p);
    if (rc) return rc;
    cudaStream_t s = ctx->stream;
    CK(P->d_segs.upload(P->h_segs, s)); CK(P->d_keys.upload(P->h_keys.keys, s));
    CK(P->d_ctr_tiles.upload(P->h_ctr_tiles, s));
    for (int v = 0; v < 4; v++) CK(P->d_tiles[v].upload(P->h_tiles[v], s));
    CK(P->d_deflate.upload(P->h_deflate, s)); CK(P->d_xz.upload(P->h_xz, s));
    if (!P->h_gcm_segs.empty()) {
        GcmDev& G = P->gcm;
        G.n_segs = (uint32_t)P->h_gcm_segs.size(); G.n_tiles = (uint32_t)P->h_gcm_tiles.size(); G.n_keys = (uint32_t)P->h_gcm_refs.size();
        CK(G.tiles.reserve(G.n_tiles + 1)); CK(G.partial.reserve(G.n_tiles + 1)); CK(G.pows.reserve(G.n_keys));
        CK(G.segs.upload(P->h_gcm_segs, s)); CK(G.tiles.upload(P->h_gcm_tiles, s)); CK(G.refs.upload(P->h_gcm_refs, s));
    }
    if (P->n_crc) {
        CK(P->d_crc_tiles.upload(P->h_crc_tiles, s)); CK(P->d_crc_first.upload(P->h_crc_first, s));
        CK(P->d_crc_expect.upload(P->h_crc_expect, s)); CK(P->d_crc_entry.upload(P->h_crc_entry, s));
        CK(P->d_crc_raw.reserve(P->h_crc_tiles.size())); CK(P->d_crc_val.reserve(P->n_crc)); CK(P->d_crc_broken.reserve(1));
    }
    CK(ctx->sync());   // the borrowed host spans may go away after this call
    return PNA_OK;
}

// assign out_off for every entry from its out_cap; (re)allocates d_out and uploads the entry table
static int decode_layout_out(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    uint64_t cur = 0;
    for (EntryRec& e : P->h_entries) {
        e.out_off = cur;
        if (e.status == ST_OK && e.out_cap != UINT64_MAX) {
            if (e.out_cap > ((uint64_t)1 << 60) || cur > ((uint64_t)1 << 60)) return PNA_E_OOM;   // checked: no wrap of the layout
            cur += align_up(e.out_cap, 16);
        }
    }
    P->out_bytes = cur;
    CK(P->d_out.reserve(cur + 256));
    // store entries: comp -> out copies in <= 256 KiB pieces
    P->h_copy.clear();
    for (uint32_t i : P->h_store) {
        const EntryRec& e = P->h_entries[i];
        uint64_t len = std::min(e.comp_len, e.out_cap);
        for (uint64_t o = 0; o < len; o += 256 * 1024) P->h_copy.push_back({e.out_off + o, e.comp_off + o, std::min<uint64_t>(256 * 1024, len - o)});
    }
    // xz: one window per XZ_WIN bytes of capacity for streams long enough to gain from it (whether a stream qualifies for the
    // chunk-parallel pass is decided on the device, from its chunk headers)
    P->h_xz_map.clear(); P->h_xz_win_begin.clear();
    if (!P->h_xz.empty()) {
        for (uint32_t k = 0; k < (uint32_t)P->h_xz.size(); k++) {
            const EntryRec& e = P->h_entries[P->h_xz[k]];
            P->h_xz_win_begin.push_back((uint32_t)P->h_xz_map.size());
            if (e.status != ST_OK || e.out_cap == UINT64_MAX) continue;
            const uint64_t nw = (e.out_cap + xz::XZ_WIN - 1) / xz::XZ_WIN;
            if (nw < 2 || nw > (1u << 16) || P->h_xz_map.size() + nw > (1u << 26)) continue;
            for (uint32_t w = 0; w < (uint32_t)nw; w++) P->h_xz_map.push_back(make_uint2(k, w));
        }
        P->h_xz_win_begin.push_back((uint32_t)P->h_xz_map.size());
        if (!P->h_xz_map.empty()) {
            CK(P->d_xz_map.upload(P->h_xz_map, ctx->stream)); CK(P->d_xz_win_begin.upload(P->h_xz_win_begin, ctx->stream));
            CK(P->d_xz_wins.reserve(P->h_xz_map.size()));
        }
    }
    // deflate: streams of the two-stage path with their literal / record arenas (sizes from the now final capacities)
    P->h_inf.clear(); P->h_deflate_big.clear();
    {
        uint64_t lit = 0, rec = 0;
        for (uint32_t i : P->h_deflate) {
            const EntryRec& e = P->h_entries[i];
            if (e.status != ST_OK) continue;
            if (e.out_cap >= 0x7FFFFFFFull) { P->h_deflate_big.push_back(i); continue; }
            P->h_inf.push_back({i, 0u, lit, rec});
            lit += align_up(e.out_cap, 16) + 16;
            rec += inf::token_rec_bound(e.out_cap);
        }
        const size_t ni = P->h_inf.size();
        if (ni) {
            CK(P->d_inf.upload(P->h_inf, ctx->stream)); CK(P->d_inf_lits.reserve(lit + 256)); CK(P->d_inf_recs.reserve(rec + 32));
            CK(P->d_inf_blocks.reserve(ni)); CK(P->d_inf_ze.reserve(ni)); CK(P->d_inf_tr.reserve(ni));
        }
        CK(P->d_deflate.upload(P->h_deflate_big, ctx->stream));   // a subset of h_deflate: fits
    }
    CK(P->d_copy.upload(P->h_copy, ctx->stream));
    CK(P->d_entries_init.upload(P->h_entries, ctx->stream));
    return PNA_OK;
}

__global__ void crc_check_kernel(const uint32_t* __restrict__ crc, const uint32_t* __restrict__ expect,
                                 const int32_t* __restrict__ entry_of, EntryRec* entries, uint32_t n, uint32_t* broken) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || crc[i] == expect[i]) return;
    atomicAdd(broken, 1u);
    if (entry_of[i] >= 0) atomicCAS(&entries[entry_of[i]].status, ST_OK, ST_INVALID_DATA);   // "broken chunk"
}
static int launch_crc(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    if (!P->n_crc) return PNA_OK;
    CK(cudaMemsetAsync(P->d_crc_broken.p, 0, sizeof(uint32_t), ctx->stream));
    const int rc = launch_chunk_crc(ctx, P->d_buf.p, P->d_crc_tiles.p, (uint32_t)P->h_crc_tiles.size(), P->d_crc_raw.p, P->d_crc_first.p,
                                    P->n_crc, P->d_crc_val.p);
    if (rc) return rc;
    crc_check_kernel<<<(P->n_crc + 127) / 128, 128, 0, ctx->stream>>>(P->d_crc_val.p, P->d_crc_expect.p, P->d_crc_entry.p, P->d_entries.p,
                                                                     P->n_crc, P->d_crc_broken.p);
    LAUNCHED();
    return PNA_OK;
}

// GCM STREAM in either direction over the segments of G, read from `src` through `segs` and written to `dst`: H and its
// powers per key, CTR and partial GHASH over the AES tiles and then the Camellia tiles, and the tags, which decryption checks
// (a mismatch fails the entry in `entries`) and encryption writes behind each segment in `dst`
template <bool DECRYPT>
static int launch_gcm(pna_ctx* ctx, const GcmDev& G, const uint8_t* src, const Segment* segs, uint8_t* dst, EntryRec* entries,
                      const DevKeys* keys) {
    if (!G.n_segs) return PNA_OK;
    const uint32_t nk = G.n_keys, ns = G.n_segs, nt = G.n_tiles, na = G.n_tiles_aes;
    gcm::gcm_setup_kernel<<<(nk + 127) / 128, 128, 0, ctx->stream>>>(G.refs.p, nk, keys, ctx->d_aes, ctx->d_cam, G.pows.p);
    LAUNCHED();
    const uint32_t cap = (uint32_t)ctx->sm_count * 3;
    if (na) {
        gcm::gcm_tiles_kernel<1, DECRYPT><<<std::min<uint32_t>((na + gcm::gcm_tile_warps<1>() - 1) / gcm::gcm_tile_warps<1>(), (uint32_t)ctx->sm_count), gcm::gcm_tile_warps<1>() * 32,
                                            gcm::gcm_tiles_smem<1>(), ctx->stream>>>(src, segs, dst, G.segs.p, G.tiles.p, na, keys, G.pows.p, ctx->d_aes, ctx->d_cam,
                                                                                     G.partial.p);
        LAUNCHED();
    }
    if (nt > na) {
        gcm::gcm_tiles_kernel<2, DECRYPT><<<std::min<uint32_t>((nt - na + gcm::gcm_tile_warps<2>() - 1) / gcm::gcm_tile_warps<2>(), cap), gcm::gcm_tile_warps<2>() * 32,
                                            gcm::gcm_tiles_smem<2>(), ctx->stream>>>(src, segs, dst, G.segs.p, G.tiles.p + na, nt - na, keys, G.pows.p, ctx->d_aes,
                                                                                     ctx->d_cam, G.partial.p + na);
        LAUNCHED();
    }
    gcm::gcm_finish_kernel<DECRYPT><<<(ns + 127) / 128, 128, 0, ctx->stream>>>(src, segs, entries, G.segs.p, ns, keys, G.pows.p, ctx->d_aes, ctx->d_cam,
                                                                               G.partial.p, DECRYPT ? nullptr : dst);
    LAUNCHED();
    return PNA_OK;
}

static int launch_cipher(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    if (const uint32_t nt = (uint32_t)P->h_ctr_tiles.size()) {
        aes_ctr_tiles_kernel<<<std::min<uint32_t>(nt, (uint32_t)ctx->sm_count), AES_CTR_THREADS, AES_CTR_TILES_SMEM, ctx->stream>>>(
            P->d_buf.p, P->d_segs.p, P->d_entries.p, P->d_ctr_tiles.p, nt, P->d_keys.p, ctx->d_aes);
        LAUNCHED();
    }
    for (int v = 0; v < 4; v++) {
        const uint32_t nt = (uint32_t)P->h_tiles[v].size();
        if (!nt) continue;
        const auto decrypt_tiles = DECRYPT_TILES[v].fn;
        decrypt_tiles<<<std::min<uint32_t>(nt, (uint32_t)ctx->sm_count * (v == 1 ? 4 : 6)), 256, DECRYPT_TILES[v].smem, ctx->stream>>>(
            P->d_buf.p, P->d_segs.p, P->d_entries.p, P->d_tiles[v].p, nt, P->d_keys.p, ctx->d_aes, ctx->d_cam);
        LAUNCHED();
    }
    return launch_gcm<true>(ctx, P->gcm, P->d_buf.p, P->d_segs.p, P->d_buf.p, P->d_entries.p, P->d_keys.p);
}

static int launch_zstd_front(pna_plan* P, bool with_count) {   // scan .. resolve
    pna_ctx* ctx = P->ctx;
    const uint32_t nz = (uint32_t)P->h_ze.size();
    if (!nz) return PNA_OK;
    if (with_count) {
        zs::zstd_count_kernel<<<(nz + 63) / 64, 64, 0, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_ze.p, nz);
        LAUNCHED();
        return PNA_OK;
    }
    zs::zstd_walk_kernel<<<(nz + 63) / 64, 64, 0, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_ze.p, nz, P->d_walk.p);
    LAUNCHED();
    if (P->n_blocks) {
        zs::zstd_fill_kernel<<<(P->n_blocks + 127) / 128, 128, 0, ctx->stream>>>(P->d_entries.p, P->d_walk.p, P->n_blocks, P->d_blocks.p);
        LAUNCHED();
        zs::zstd_parse_kernel<<<(P->n_blocks + 127) / 128, 128, 0, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_blocks.p, P->n_blocks);
        LAUNCHED();
    }
    zs::zstd_resolve_kernel<<<(nz + 3) / 4, 128, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, nz, P->d_blocks.p);   // warp per entry
    LAUNCHED();
    zs::zstd_order_kernel<<<1, 1024, 0, ctx->stream>>>(P->d_entries.p, P->d_blocks.p, P->n_blocks, P->d_seq_order.p, P->d_lit_order.p,
                                                      P->d_counts.p);
    LAUNCHED();
    return PNA_OK;
}
static int launch_zstd_seq(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    if (P->h_ze.empty() || !P->n_blocks) return PNA_OK;
    const uint32_t per_cta = zs::SEQ_SLOTS * zs::SEQ_WARPS;
    const uint32_t grid = std::min<uint32_t>((P->n_blocks + per_cta - 1) / per_cta, (uint32_t)ctx->sm_count);
    zs::zstd_seq_kernel<<<grid, 32 * zs::SEQ_WARPS, zs::SEQ_SMEM_BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_blocks.p, P->d_seq_order.p,
                                                                      P->d_counts.p, P->d_seq_base.p, P->d_seqs.p);
    LAUNCHED();
    return PNA_OK;
}
static int launch_zstd_lit(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    if (P->h_ze.empty() || !P->n_blocks) return PNA_OK;
    const uint32_t grid = std::min<uint32_t>((P->n_blocks + zs::LIT_SLOTS - 1) / zs::LIT_SLOTS, (uint32_t)ctx->sm_count * 3);
    zs::zstd_lit_kernel<<<grid, 32, zs::LIT_SMEM_BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_blocks.p, P->d_lit_order.p,
                                                                      P->d_counts.p, P->d_lit_base.p, P->d_lits.p);
    LAUNCHED();
    return PNA_OK;
}
static int launch_zstd_prefix(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    const uint32_t nz = (uint32_t)P->h_ze.size();
    if (!nz) return PNA_OK;
    zs::zstd_prefix_kernel<<<(nz + 3) / 4, 128, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, nz, P->d_blocks.p);   // warp per entry
    LAUNCHED();
    return PNA_OK;
}
// Entries taken block-parallel inside their frames: per segment  scan -> expand -> pointer-jumping rounds -> gather.
// The rounds after the one that found every pointer at a root return at once (flag of the previous round), so the fixed
// launch sequence needs no host round trip.
static int launch_zstd_pj(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    const uint32_t ns = (uint32_t)P->h_pj_segs.size();
    if (!ns) return PNA_OK;
    CK(cudaMemsetAsync(P->d_pj_flags.p, 0, (size_t)ns * zs::PJ_MAX_ROUNDS * sizeof(uint32_t), ctx->stream));
    const uint32_t jump_grid = (uint32_t)ctx->sm_count * 8;
    for (uint32_t s = 0; s < ns; s++) {
        const uint32_t nb = P->h_pj_segs[s].blk_count;
        uint32_t* flags = P->d_pj_flags.p + (size_t)s * zs::PJ_MAX_ROUNDS;
        zs::pj_scan_kernel<<<(nb + 7) / 8, 256, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, P->d_pj_segs.p, s, P->d_blocks.p, P->d_seqs.p, P->d_pj_cpos.p);
        LAUNCHED();
        zs::pj_expand_kernel<<<dim3(zs::PJ_EXPAND_X, nb), 256, 0, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_ze.p, P->d_pj_segs.p, s, P->d_blocks.p,
                                                                                P->d_lits.p, P->d_seqs.p, P->d_pj_cpos.p, P->d_out.p, P->d_pj_ptr.p);
        LAUNCHED();
        uint8_t* tiles[2] = {P->d_pj_tiles.p, P->d_pj_tiles.p + P->pj_tile_stride};
        zs::pj_chase_kernel<<<jump_grid, 256, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, P->d_pj_segs.p, s, P->d_blocks.p, P->d_pj_ptr.p, tiles[0]);
        LAUNCHED();
        for (int r = 0; r < zs::PJ_MAX_ROUNDS; r++) {
            zs::pj_jump_kernel<<<jump_grid, 256, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, P->d_pj_segs.p, s, P->d_blocks.p, P->d_pj_ptr.p, flags, r,
                                                                   tiles[r & 1], tiles[(r + 1) & 1]);
            LAUNCHED();
        }
        zs::pj_gather_kernel<<<jump_grid, 256, 0, ctx->stream>>>(P->d_entries.p, P->d_ze.p, P->d_pj_segs.p, s, P->d_blocks.p, P->d_pj_ptr.p, flags, P->d_out.p);
        LAUNCHED();
    }
    return PNA_OK;
}
static int launch_zstd_lz_on(pna_plan* P, const zs::ZEntry* ze, const uint32_t* order, const zs::LzUnit* units, uint32_t nz,
                             const zs::ZBlock* blocks, const uint8_t* lits, const zs::SeqRec* seqs) {
    pna_ctx* ctx = P->ctx;
    if (!nz) return PNA_OK;
    // one CTA per unit (frame), longest streams first.  Fewer units than half the SMs (a reference-written solid archive is ONE
    // frame): the 16-warp variant with the 128 KiB window; otherwise 4 warps per unit, 7 units per SM.  In between -- up to four
    // waves of large units (measured on 4 MiB entries: 16 warps x 1 unit per SM beat 4 warps x 7 up to ~600 units; 256 entries
    // 10.7 -> 5.8 ms) -- the 16-warp variant too, because a unit is serial and more warps per unit is the only parallelism left.
    const char* force = getenv("PNA_LZ_VARIANT");
    const bool big = force ? force[0] == 'b'
                           : nz * 2 <= (uint32_t)ctx->sm_count || (units && nz <= 4u * (uint32_t)ctx->sm_count && P->lz_avg_unit_comp >= (256u << 10));
    if (big)
        zs::zstd_lz_kernel<zs::LzBig><<<nz, zs::LzBig::T, zs::LzBig::BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, ze, order, units, nz, blocks, lits,
                                                                                            seqs, P->d_out.p);
    else
        zs::zstd_lz_kernel<zs::LzSmall><<<nz, zs::LzSmall::T, zs::LzSmall::BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, ze, order, units, nz, blocks,
                                                                                                lits, seqs, P->d_out.p);
    LAUNCHED();
    return PNA_OK;
}
// size_only (before the output layout exists): one lane per stream counts the decoded length of EVERY deflate entry.
// Otherwise: tokens -> LZ -> Adler for the two-stage streams, the bits-to-bytes kernel for the >= 2 GiB ones.
static int launch_inflate(pna_plan* P, int size_only) {
    pna_ctx* ctx = P->ctx;
    const uint32_t nx = (uint32_t)P->h_xz.size();
    if (nx) {   // xz: a warp per stream (kernels_xz.cuh); sizing reads the chunk headers only
        const uint32_t nw = size_only ? 0u : (uint32_t)P->h_xz_map.size();
        if (nw) {   // streams made of independent chunks (this library's writer): a warp per 32 KiB window first
            xz::xz_window_kernel<<<nw, 32, xz::XZ_WIN_SMEM_BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_xz.p, P->d_xz_map.p, nw, P->d_out.p, P->d_xz_wins.p);
            LAUNCHED();
        }
        xz::xz_decode_kernel<<<nx, 32, xz::XZ_SMEM_BYTES, ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_xz.p, nx, P->d_out.p, size_only,
                                                                         nw ? P->d_xz_win_begin.p : nullptr, nw ? P->d_xz_wins.p : nullptr);
        LAUNCHED();
    }
    if (size_only) {
        const uint32_t nd = (uint32_t)P->h_deflate.size();
        if (!nd) return PNA_OK;
        std::vector<inf::InfStream> all(nd);
        for (uint32_t k = 0; k < nd; k++) all[k] = {P->h_deflate[k], 0u, 0ull, 0ull};
        CK(P->d_inf.upload(all, ctx->stream));
        inf::inflate_tokens_kernel<<<(nd + inf::TOKEN_CTA - 1) / inf::TOKEN_CTA, inf::TOKEN_CTA, inf::TOKEN_SMEM_BYTES, ctx->stream>>>(
            P->d_buf.p, P->d_entries.p, P->d_inf.p, nd, nullptr, nullptr, nullptr, nullptr, nullptr, 1);
        LAUNCHED();
        CK(ctx->sync());   // `all` is a local
        return PNA_OK;
    }
    const uint32_t ni = (uint32_t)P->h_inf.size(), nb = (uint32_t)P->h_deflate_big.size();
    if (ni) {
        inf::inflate_tokens_kernel<<<(ni + inf::TOKEN_CTA - 1) / inf::TOKEN_CTA, inf::TOKEN_CTA, inf::TOKEN_SMEM_BYTES, ctx->stream>>>(
            P->d_buf.p, P->d_entries.p, P->d_inf.p, ni, P->d_inf_lits.p, P->d_inf_recs.p, P->d_inf_blocks.p, P->d_inf_ze.p, P->d_inf_tr.p, 0);
        LAUNCHED();
        int rc = launch_zstd_lz_on(P, P->d_inf_ze.p, nullptr, nullptr, ni, P->d_inf_blocks.p, P->d_inf_lits.p, P->d_inf_recs.p);
        if (rc) return rc;
        inf::inflate_adler_kernel<<<(ni + 7) / 8, 256, 0, ctx->stream>>>(P->d_entries.p, P->d_inf.p, P->d_inf_tr.p, ni, P->d_out.p);
        LAUNCHED();
    }
    if (nb) {
        inf::inflate_kernel<<<(nb + inf::INFLATE_CTA - 1) / inf::INFLATE_CTA, 32 * inf::INFLATE_CTA, sizeof(inf::Tables) * inf::INFLATE_CTA,
                              ctx->stream>>>(P->d_buf.p, P->d_entries.p, P->d_deflate.p, nb, P->d_out.p, 0);
        LAUNCHED();
    }
    return PNA_OK;
}
static int launch_zstd_pj(pna_plan* P);
static int launch_zstd_lz(pna_plan* P) {
    int rc = launch_zstd_lz_on(P, P->d_ze.p, P->d_lz_order.p, P->d_lz_units.p, P->n_lz_units, P->d_blocks.p, P->d_lits.p, P->d_seqs.p);
    return rc ? rc : launch_zstd_pj(P);
}
static int launch_store(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    const uint32_t nc = (uint32_t)P->h_copy.size();
    if (!nc) return PNA_OK;
    const uint32_t grid = std::min<uint32_t>((nc + 7) / 8, (uint32_t)ctx->sm_count * 8);
    copy_jobs_kernel<<<grid, 256, 0, ctx->stream>>>(P->d_out.p, P->d_buf.p, P->d_copy.p, nc);
    LAUNCHED();
    return PNA_OK;
}

// One-time preparation: learn block / literal / sequence counts (and output sizes when no hint was
// given), allocate, lay out.  Runs the front kernels once; launch_all() re-runs everything.
static int decode_prepare(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    int rc;
    const uint32_t nz = (uint32_t)P->h_ze.size();
    CK(P->d_entries.upload(P->h_entries, ctx->stream));
    if ((rc = launch_crc(P))) return rc;
    if ((rc = launch_cipher(P))) return rc;
    if (nz) {
        CK(P->d_ze.upload(P->h_ze, ctx->stream));
        // LZ stage order: longest compressed streams first (one CTA per entry, dispatched in grid order)
        std::vector<uint32_t> lz_order(nz);
        for (uint32_t i = 0; i < nz; i++) lz_order[i] = i;
        std::stable_sort(lz_order.begin(), lz_order.end(), [&](uint32_t a, uint32_t b) {
            return P->h_entries[P->h_ze[a].entry].comp_len > P->h_entries[P->h_ze[b].entry].comp_len; });
        if ((rc = launch_zstd_front(P, true))) return rc;
        CK(cudaMemcpyAsync(P->h_ze.data(), P->d_ze.p, nz * sizeof(zs::ZEntry), cudaMemcpyDeviceToHost, ctx->stream));
        CK(ctx->sync());
        uint64_t nb = 0;
        for (auto& z : P->h_ze) { z.blk_begin = (uint32_t)nb; nb += z.blk_count; }
        if (nb > 0xFFFFFFF0ull) return PNA_E_OOM;
        P->n_blocks = (uint32_t)nb;
        CK(P->d_blocks.reserve(nb)); CK(P->d_walk.reserve(nb));
        CK(P->d_seq_order.reserve(nb)); CK(P->d_lit_order.reserve(nb)); CK(P->d_counts.reserve(8));
        CK(P->d_ze.upload(P->h_ze, ctx->stream));
        if ((rc = launch_zstd_front(P, false))) return rc;
        CK(cudaMemcpyAsync(P->h_ze.data(), P->d_ze.p, nz * sizeof(zs::ZEntry), cudaMemcpyDeviceToHost, ctx->stream));
        CK(ctx->sync());
        uint64_t lit = 0, seq = 0, nu = 0;
        std::vector<uint64_t> lb(P->n, 0), sb(P->n, 0);
        for (auto& z : P->h_ze) {
            z.lit_base = lit; z.seq_base = seq;
            lb[z.entry] = lit; sb[z.entry] = seq;
            lit += z.lit_total; seq += z.seq_total;
            z.unit_begin = (uint32_t)nu; nu += z.n_frames;
        }
        if (nu > 0xFFFFFFF0ull) return PNA_E_OOM;
        // LZ units = frames; dispatched entry by entry in the longest-stream-first order, an entry's frames in stream order
        P->n_lz_units = (uint32_t)nu;   // (reduced to the units of the CTA-per-frame kernel below)
        {
            uint64_t zc = 0;
            for (const auto& z : P->h_ze) zc += P->h_entries[z.entry].comp_len;
            P->lz_avg_unit_comp = nu ? zc / nu : 0;
        }
        // Entries of very many blocks (a reference-written solid archive: ONE frame over every file) leave the CTA-per-frame
        // kernel with a single busy SM: they are decoded block-parallel by pointer jumping instead (kernels_zstd_pj.cuh), as
        // long as there are few of them -- with many large entries the frames themselves are the parallelism.
        const char* pj_env = getenv("PNA_LZ_PJ_MIN_BLOCKS");
        const uint32_t pj_min = pj_env ? (uint32_t)atoi(pj_env) : 512u;
        std::vector<uint8_t> is_pj(nz, 0);
        {
            uint32_t n_big = 0;
            for (uint32_t zi = 0; zi < nz; zi++) if (pj_min && P->h_ze[zi].blk_count >= pj_min) n_big++;
            if (n_big && (n_big <= 16 || pj_env))
                for (uint32_t zi = 0; zi < nz; zi++) if (P->h_ze[zi].blk_count >= pj_min && P->h_ze[zi].blk_count > 0) is_pj[zi] = 1;
        }
        P->h_pj_segs.clear(); P->pj_max_blocks = 0;
        for (uint32_t zi = 0; zi < nz; zi++) {
            if (!is_pj[zi]) continue;
            const auto& z = P->h_ze[zi];
            for (uint32_t b0 = 0; b0 < z.blk_count; b0 += zs::PJ_SEG_BLOCKS) {
                const uint32_t nbk = std::min<uint32_t>(zs::PJ_SEG_BLOCKS, z.blk_count - b0);
                P->h_pj_segs.push_back({zi, z.blk_begin + b0, nbk, 0u});
                P->pj_max_blocks = std::max(P->pj_max_blocks, nbk);
            }
        }
        if (!P->h_pj_segs.empty()) {
            CK(P->d_pj_segs.upload(P->h_pj_segs, ctx->stream));
            CK(P->d_pj_ptr.reserve((size_t)P->pj_max_blocks * zs::BLOCK_MAX + 64));
            CK(P->d_pj_cpos.reserve((size_t)P->pj_max_blocks * zs::PJ_MAX_CHUNKS));
            CK(P->d_pj_flags.reserve(P->h_pj_segs.size() * zs::PJ_MAX_ROUNDS));
            P->pj_tile_stride = align_up((uint64_t)P->pj_max_blocks * zs::BLOCK_MAX / 1024 + 64, 256);
            CK(P->d_pj_tiles.reserve(2 * P->pj_tile_stride));
        }
        std::vector<uint32_t> unit_order;
        unit_order.reserve(nu);
        for (uint32_t zi : lz_order) {
            if (is_pj[zi]) continue;
            for (uint32_t f = 0; f < P->h_ze[zi].n_frames; f++) unit_order.push_back(P->h_ze[zi].unit_begin + f);
        }
        CK(P->d_lz_order.reserve(nu + 1)); CK(P->d_lz_units.reserve(nu + 1));
        CK(P->d_lz_order.upload(unit_order, ctx->stream));
        const uint32_t n_regular_units = (uint32_t)unit_order.size();
        P->lit_total = lit; P->seq_total = seq;
        CK(P->d_lits.reserve(lit + 256));
        CK(P->d_seqs.reserve(seq + 32));
        CK(P->d_lit_base.upload(lb, ctx->stream)); CK(P->d_seq_base.upload(sb, ctx->stream));
        CK(P->d_ze.upload(P->h_ze, ctx->stream));
        zs::zstd_units_kernel<<<(nz + 127) / 128, 128, 0, ctx->stream>>>(P->d_ze.p, nz, P->d_blocks.p, P->d_lz_units.p);
        LAUNCHED();
        CK(ctx->sync());   // lb/sb/unit_order are locals
        P->n_lz_units = n_regular_units;
    }
    if (P->need_sizing) {
        // exact sizes: zstd from the entropy+prefix stages, deflate from a count-only pass, store = comp_len
        if ((rc = launch_zstd_seq(P))) return rc;
        if ((rc = launch_zstd_lit(P))) return rc;
        if ((rc = launch_zstd_prefix(P))) return rc;
        if ((rc = launch_inflate(P, 1))) return rc;
        P->sized_entropy = true;
        std::vector<EntryRec> dev(P->n);
        CK(cudaMemcpyAsync(dev.data(), P->d_entries.p, P->n * sizeof(EntryRec), cudaMemcpyDeviceToHost, ctx->stream));
        CK(ctx->sync());
        for (uint32_t i = 0; i < P->n; i++) {
            EntryRec& e = P->h_entries[i];
            if (e.status != ST_OK || e.out_cap != UINT64_MAX) continue;
            if (dev[i].status != ST_OK) { e.out_cap = 0; continue; }   // will fail again in the real run
            e.out_cap = e.compression == PNA_COMPRESSION_NO ? dev[i].comp_len : dev[i].out_len;
            if (e.compression == PNA_COMPRESSION_NO) e.comp_len = dev[i].comp_len;
        }
    }
    if ((rc = decode_layout_out(P))) return rc;
    CK(ctx->sync());
    P->prepared = true;
    return PNA_OK;
}

__global__ void set_layout_kernel(EntryRec* entries, const uint64_t* __restrict__ off_cap, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    entries[i].out_off = off_cap[2 * i];
    entries[i].out_cap = off_cap[2 * i + 1];
}

#define STAGE(i) do { if (P->ev_ready) CK(cudaEventRecord(P->ev[i], ctx->stream)); } while (0)
// the plan's stage-timing events, on its first run: from the context's pool (~pna_plan gives them back) or new
static int lease_stage_events(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    if (P->ev_ready) return PNA_OK;
    for (auto& e : P->ev) {
        if (!ctx->ev_pool.empty()) { e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
        else CK(cudaEventCreate(&e));
    }
    P->ev_ready = true;
    return PNA_OK;
}
// fresh = true: full pipeline from the pristine entry table (every run after the first).
// fresh = false: continue right after decode_prepare(), which already decrypted and scanned (and, when it had
// to size outputs, entropy-decoded) on the live table -- so a one-shot pna_cuda_decode_batch does no work twice.
static int decode_launch_all(pna_plan* P, bool fresh) {
    pna_ctx* ctx = P->ctx;
    int rc;
    const uint64_t l0 = ctx->launches;
    if ((rc = lease_stage_events(P))) return rc;
    if (fresh) {
        CK(cudaMemcpyAsync(P->d_entries.p, P->d_entries_init.p, P->n * sizeof(EntryRec), cudaMemcpyDeviceToDevice, ctx->stream));
        STAGE(0);
        if ((rc = launch_crc(P))) return rc;
        STAGE(1);
        if ((rc = launch_cipher(P))) return rc;
        STAGE(2);
        if ((rc = launch_zstd_front(P, false))) return rc;
    } else {
        std::vector<uint64_t> oc(2 * (size_t)P->n);
        for (uint32_t i = 0; i < P->n; i++) { oc[2 * i] = P->h_entries[i].out_off; oc[2 * i + 1] = P->h_entries[i].out_cap; }
        CK(P->d_layout.upload(oc, ctx->stream));
        set_layout_kernel<<<(P->n + 127) / 128, 128, 0, ctx->stream>>>(P->d_entries.p, P->d_layout.p, P->n);
        LAUNCHED();
        CK(ctx->sync());   // oc is a local
        STAGE(0); STAGE(1); STAGE(2);
    }
    STAGE(3);
    const bool entropy = fresh || !P->sized_entropy;   // decode_prepare's sizing pass leaves the entropy stages done
    if (entropy && (rc = launch_zstd_seq(P))) return rc;
    STAGE(4);
    if (entropy && (rc = launch_zstd_lit(P))) return rc;
    STAGE(5);
    if (entropy && (rc = launch_zstd_prefix(P))) return rc;
    STAGE(6);
    if ((rc = launch_zstd_lz(P))) return rc;
    STAGE(7);
    if ((rc = launch_inflate(P, 0))) return rc;
    STAGE(8);
    if ((rc = launch_store(P))) return rc;
    STAGE(9);
    P->ev_recorded = true;
    if (fresh) P->launches_per_run = ctx->launches - l0;
    return PNA_OK;
}

static int decode_plan_create_ex(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, const uint64_t* caps, const CrcReq* crc,
                                 pna_plan** plan) {
    if (!ctx || !plan || (!descs && n)) return PNA_E_BAD_ARG;
    *plan = nullptr;
    if (!ctx->devs.empty()) return multi::decode_plan_create(ctx, descs, n, crc, plan);   // (caps only come from pna_cuda_decode_batch, which shards first)
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    pna_plan* P = new pna_plan();
    int rc = decode_plan_build(ctx, descs, n, caps, crc, P);
    if (rc) { delete P; return rc; }
    *plan = P;
    return PNA_OK;
}
extern "C" int pna_cuda_decode_plan_create(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, pna_plan** plan) {
    return decode_plan_create_ex(ctx, descs, n, nullptr, nullptr, plan);
}
extern "C" int pna_cuda_decode_plan_create_crc(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, const pna_span* crc_spans,
                                               const uint32_t* crc_expect, const int32_t* crc_entry, uint32_t n_spans,
                                               pna_plan** plan) {
    if (n_spans && (!crc_spans || !crc_expect || !crc_entry)) return PNA_E_BAD_ARG;
    for (uint32_t i = 0; i < n_spans; i++) if (crc_entry[i] >= (int64_t)n) return PNA_E_BAD_ARG;
    CrcReq rq{crc_spans, crc_expect, crc_entry, n_spans, nullptr, 0};
    return decode_plan_create_ex(ctx, descs, n, nullptr, &rq, plan);
}
extern "C" int pna_cuda_decode_plan_create_in_image(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, const uint8_t* image,
                                                    uint64_t image_len, const pna_span* crc_spans, const uint32_t* crc_expect,
                                                    const int32_t* crc_entry, uint32_t n_spans, pna_plan** plan) {
    if (n_spans && (!crc_spans || !crc_expect || !crc_entry)) return PNA_E_BAD_ARG;
    if (!image && image_len) return PNA_E_BAD_ARG;
    for (uint32_t i = 0; i < n_spans; i++) if (crc_entry[i] >= (int64_t)n) return PNA_E_BAD_ARG;
    CrcReq rq{crc_spans, crc_expect, crc_entry, n_spans, image, image_len};
    return decode_plan_create_ex(ctx, descs, n, nullptr, &rq, plan);
}
extern "C" int pna_cuda_plan_crc_results(pna_plan* P, uint32_t* crc_out, uint32_t* n_broken) {
    if (!P) return PNA_E_BAD_ARG;
    if (P->multi) return multi::plan_crc_results(P, crc_out, n_broken);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (n_broken) *n_broken = 0;
    if (!P->n_crc || !P->prepared) return PNA_OK;
    if (crc_out) CK(cudaMemcpyAsync(crc_out, P->d_crc_val.p, P->n_crc * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (n_broken) CK(cudaMemcpyAsync(n_broken, P->d_crc_broken.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    return PNA_OK;
}
extern "C" int pna_cuda_decode_plan_run(pna_plan* P) {
    if (!P || P->kind != 0) return PNA_E_BAD_ARG;
    if (P->multi) return multi::decode_plan_run(P);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    if (!P->prepared) {
        int rc = decode_prepare(P);
        if (rc) return rc;
        return decode_launch_all(P, false);
    }
    return decode_launch_all(P, true);
}
// An entry's status and decoded length after a run, from its host record `h` and its device record `d`: a host-side
// rejection first, then the device's status, then the plan's capacity.  The length is 0 unless the status is OK or NOSPACE.
static int32_t decode_result(const EntryRec& h, const EntryRec& d, uint64_t* len) {
    int32_t st = d.status;
    uint64_t l = d.compression == PNA_COMPRESSION_NO ? d.comp_len : d.out_len;
    if (h.status != ST_OK) { st = h.status; l = 0; }
    if (st == ST_OK && l > d.out_cap) st = ST_NOSPACE;
    *len = (st == ST_OK || st == ST_NOSPACE) ? l : 0;
    return st;
}
extern "C" int pna_cuda_decode_plan_fetch(pna_plan* P, pna_buf* out, int32_t* status) {
    if (!P || P->kind != 0 || ((!out || !status) && P->n)) return PNA_E_BAD_ARG;
    if (P->multi) return multi::decode_plan_fetch(P, out, status);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    if (!P->prepared) return PNA_E_BAD_ARG;
    std::vector<EntryRec> dev(P->n);
    CK(cudaMemcpyAsync(dev.data(), P->d_entries.p, P->n * sizeof(EntryRec), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    uint64_t plain = 0;
    // D2H: entries whose host buffers mirror the device layout (same distance between starts, inside the previous
    // buffer's capacity) travel in ONE cudaMemcpyAsync -- a million small files must not mean a million copies
    uint8_t* run_host = nullptr;
    uint64_t run_dev = 0, run_len = 0;
    auto flush_run = [&]() -> int {
        if (run_len) CK(cudaMemcpyAsync(run_host, P->d_out.p + run_dev, run_len, cudaMemcpyDeviceToHost, ctx->stream));
        run_len = 0;
        return PNA_OK;
    };
    uint32_t prev = UINT32_MAX;
    for (uint32_t i = 0; i < P->n; i++) {
        const EntryRec& e = dev[i];
        uint64_t len;
        int32_t st = decode_result(P->h_entries[i], e, &len);
        if (st == ST_OK && len > out[i].cap) st = ST_NOSPACE;
        out[i].len = len;
        status[i] = st;
        if (st == ST_OK && len) {
            bool merged = false;
            if (run_len && prev != UINT32_MAX) {
                const uint64_t d_host = (uint64_t)(out[i].ptr - out[prev].ptr), d_dev = e.out_off - dev[prev].out_off;
                if (out[i].ptr > out[prev].ptr && d_host == d_dev && d_host <= out[prev].cap && run_dev + run_len <= e.out_off &&
                    run_host + (e.out_off - run_dev) == out[i].ptr) {
                    run_len = e.out_off - run_dev + len;
                    merged = true;
                }
            }
            if (!merged) {
                int rc = flush_run();
                if (rc) return rc;
                run_host = out[i].ptr; run_dev = e.out_off; run_len = len;
            }
            prev = i;
            plain += len;
        }
    }
    {
        int rc = flush_run();
        if (rc) return rc;
    }
    P->plain_bytes = plain;
    CK(ctx->sync());
    return PNA_OK;
}
extern "C" int pna_cuda_decode_plan_lengths(pna_plan* P, uint64_t* out_len, int32_t* status) {
    if (!P || P->kind != 0 || ((!out_len || !status) && P->n)) return PNA_E_BAD_ARG;
    if (P->multi) return multi::decode_plan_lengths(P, out_len, status);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    if (!P->prepared) return PNA_E_BAD_ARG;
    std::vector<EntryRec> dev(P->n);
    CK(cudaMemcpyAsync(dev.data(), P->d_entries.p, P->n * sizeof(EntryRec), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    P->h_out_len.resize(P->n);
    for (uint32_t i = 0; i < P->n; i++) {
        status[i] = decode_result(P->h_entries[i], dev[i], &out_len[i]);
        P->h_out_len[i] = status[i] == ST_OK ? out_len[i] : 0;
    }
    return PNA_OK;
}
// the decoded bytes of `entry` as they sit in HBM after a run (lengths must have been queried)
static int plan_entry_out(pna_plan* P, uint32_t entry, const uint8_t** base, uint64_t* len) {
    if (!P || P->kind != 0 || entry >= P->n || !P->prepared || P->h_out_len.size() != P->n) return PNA_E_BAD_ARG;
    *base = P->d_out.p + P->h_entries[entry].out_off;
    *len = P->h_out_len[entry];
    return PNA_OK;
}
extern "C" int pna_cuda_decode_plan_crc32_out(pna_plan* P, uint32_t entry, const uint64_t* span_off, const uint64_t* span_len,
                                              uint32_t n, uint32_t* crc_out) {
    if (P && P->multi) P = multi::route(P, &entry);
    const uint8_t* base = nullptr;
    uint64_t len = 0;
    int rc = plan_entry_out(P, entry, &base, &len);
    if (rc) return rc;
    if (n == 0) return PNA_OK;
    if (!span_off || !span_len || !crc_out) return PNA_E_BAD_ARG;
    for (uint32_t i = 0; i < n; i++) if (span_off[i] > len || span_len[i] > len - span_off[i]) return PNA_E_BAD_ARG;
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    std::vector<uint64_t> off(span_off, span_off + n);
    return crc_run(ctx, base, off, span_len, n, crc_out);
}
extern "C" int pna_cuda_decode_plan_fetch_ranges(pna_plan* P, uint32_t entry, const uint64_t* src_off, const uint64_t* len,
                                                 uint8_t* const* dst, uint32_t n) {
    if (P && P->multi) P = multi::route(P, &entry);
    const uint8_t* base = nullptr;
    uint64_t total = 0;
    int rc = plan_entry_out(P, entry, &base, &total);
    if (rc) return rc;
    if (n == 0) return PNA_OK;
    if (!src_off || !len || !dst) return PNA_E_BAD_ARG;
    for (uint32_t i = 0; i < n; i++) if (src_off[i] > total || len[i] > total - src_off[i] || (len[i] && !dst[i])) return PNA_E_BAD_ARG;
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    // ranges that continue each other on both sides travel in one copy
    uint64_t run_src = 0, run_len = 0;
    uint8_t* run_dst = nullptr;
    for (uint32_t i = 0; i < n; i++) {
        if (!len[i]) continue;
        if (run_len && src_off[i] == run_src + run_len && dst[i] == run_dst + run_len) { run_len += len[i]; continue; }
        if (run_len) CK(cudaMemcpyAsync(run_dst, base + run_src, run_len, cudaMemcpyDeviceToHost, ctx->stream));
        run_src = src_off[i]; run_len = len[i]; run_dst = dst[i];
    }
    if (run_len) CK(cudaMemcpyAsync(run_dst, base + run_src, run_len, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    return PNA_OK;
}
extern "C" int pna_cuda_plan_stats(pna_plan* P, uint64_t* stream_bytes, uint64_t* plain_bytes, uint64_t* launches_per_run) {
    if (!P) return PNA_E_BAD_ARG;
    if (P->multi) { multi::sum_stats(P, stream_bytes, plain_bytes, launches_per_run, false); return PNA_OK; }
    if (stream_bytes) *stream_bytes = P->stream_bytes;
    if (plain_bytes) *plain_bytes = P->plain_bytes;
    if (launches_per_run) *launches_per_run = P->launches_per_run;
    return PNA_OK;
}
extern "C" int pna_cuda_plan_counts(pna_plan* P, uint64_t* n_blocks, uint64_t* n_sequences, uint64_t* literal_bytes) {
    if (!P) return PNA_E_BAD_ARG;
    if (P->multi) { multi::sum_stats(P, n_blocks, n_sequences, literal_bytes, true); return PNA_OK; }
    if (n_blocks) *n_blocks = P->n_blocks;
    if (n_sequences) *n_sequences = P->seq_total;
    if (literal_bytes) *literal_bytes = P->lit_total;
    return PNA_OK;
}
extern "C" int pna_cuda_plan_stage_ms(pna_plan* P, float* ms, uint32_t cap) {
    if (!P) return -1;
    if (P->multi) return multi::stage_ms(P, ms, cap);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!P->ev_recorded) return 0;
    if (cudaEventSynchronize(P->ev[PNA_N_STAGES]) != cudaSuccess) return -1;
    for (int i = 0; i < PNA_N_STAGES && (uint32_t)i < cap; i++) {
        float t = 0;
        cudaEventElapsedTime(&t, P->ev[i], P->ev[i + 1]);
        ms[i] = t;
    }
    return PNA_N_STAGES;
}
extern "C" const char* pna_cuda_stage_name(uint32_t i) { return i < (uint32_t)PNA_N_STAGES ? PNA_STAGE_NAMES[i] : ""; }
extern "C" void pna_cuda_plan_destroy(pna_plan* P) {
    if (!P) return;
    if (P->multi) { multi::plan_destroy(P); return; }
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    ctx->sync();
    delete P;
}
extern "C" int pna_cuda_decode_batch(pna_ctx* ctx, const pna_decode_desc* descs, uint32_t n, pna_buf* out, int32_t* status) {
    if (!ctx || ((!descs || !out || !status) && n)) return PNA_E_BAD_ARG;
    if (n == 0) return PNA_OK;
    if (!ctx->devs.empty()) return multi::decode_batch(ctx, descs, n, out, status);
    std::vector<uint64_t> caps(n);
    for (uint32_t i = 0; i < n; i++) caps[i] = out[i].cap;
    pna_plan* P = nullptr;
    int rc = decode_plan_create_ex(ctx, descs, n, caps.data(), nullptr, &P);
    if (rc) return rc;
    rc = pna_cuda_decode_plan_run(P);
    if (rc == PNA_OK) rc = pna_cuda_decode_plan_fetch(P, out, status);
    pna_cuda_plan_destroy(P);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// block-cipher test hook
// GCM STREAM key schedule, host only (entry/read.rs:105-139 order of checks; aead.rs:134-208)
extern "C" int32_t pna_cuda_gcm_stream_key(const uint8_t k_master[32], const uint8_t* stream_header, uint64_t stream_header_len,
                                           const uint8_t header_type[4], const uint8_t* header_data, uint64_t header_len,
                                           const uint8_t* phsf, uint64_t phsf_len, uint8_t out_key[32]) {
    if (!k_master || !header_type || !out_key || (!stream_header && stream_header_len) || (!header_data && header_len) || (!phsf && phsf_len))
        return PNA_E_BAD_ARG;
    if (stream_header_len < aead::STREAM_HEADER_LEN) return PNA_E_INVALID_DATA;   // "datastream shorter than the stream header"
    const uint32_t seg = (uint32_t)stream_header[39] << 24 | (uint32_t)stream_header[40] << 16 | (uint32_t)stream_header[41] << 8 | stream_header[42];
    if (seg == 0 || seg > gcm::GCM_MAX_SEGMENT) return PNA_E_INVALID_DATA;       // "segment size out of range"
    uint8_t kc[32], diff = 0;
    aead::key_confirmation(k_master, kc);
    for (int i = 0; i < 32; i++) diff |= (uint8_t)(kc[i] ^ stream_header[43 + i]);
    if (diff) return PNA_E_INVALID_DATA;                                         // AeadError::KeyMismatch
    aead::derive_stream_key(k_master, stream_header, header_type, header_data, header_len, phsf, phsf_len, out_key);
    return PNA_OK;
}
extern "C" int32_t pna_cuda_gcm_stream_header(const uint8_t k_master[32], const uint8_t salt[32], const uint8_t nonce_prefix[7],
                                              uint32_t segment_size, uint8_t out_header[75]) {
    if (!k_master || !salt || !nonce_prefix || !out_header) return PNA_E_BAD_ARG;
    if (segment_size == 0 || segment_size > gcm::GCM_MAX_SEGMENT) return PNA_E_INVALID_INPUT;
    memcpy(out_header, salt, 32);
    memcpy(out_header + 32, nonce_prefix, 7);
    out_header[39] = (uint8_t)(segment_size >> 24); out_header[40] = (uint8_t)(segment_size >> 16);
    out_header[41] = (uint8_t)(segment_size >> 8); out_header[42] = (uint8_t)segment_size;
    aead::key_confirmation(k_master, out_header + 43);
    return PNA_OK;
}

extern "C" int pna_cuda_ecb(pna_ctx* ctx, int encryption, int encrypt, const uint8_t key[32], const uint8_t* in, uint64_t n_bytes,
                            uint8_t* out) {
    if (!ctx || !key || (!in && n_bytes) || (!out && n_bytes)) return PNA_E_BAD_ARG;
    if (encryption != 1 && encryption != 2) return PNA_E_BAD_ARG;
    if (!ctx->devs.empty()) return pna_cuda_ecb(ctx->devs[0], encryption, encrypt, key, in, n_bytes, out);
    const uint64_t nb = n_bytes / 16;
    if (!nb) return PNA_OK;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    const DevKeys dk = expand_key(ctx, (uint8_t)encryption, key);
    DevArr<uint8_t> d_in, d_out; DevArr<DevKeys> d_key;
    CK(d_in.reserve(nb * 16 + 64)); CK(d_out.reserve(nb * 16));
    CK(cudaMemcpyAsync(d_in.p, in, nb * 16, cudaMemcpyHostToDevice, ctx->stream));
    CK(d_key.upload(&dk, 1, ctx->stream));
    const uint32_t grid = (uint32_t)std::min<uint64_t>((nb + 255) / 256, (uint64_t)ctx->sm_count * 4);
    ecb_kernel<<<grid, 256, ECB_SMEM, ctx->stream>>>(encryption, encrypt, d_key.p, ctx->d_aes, ctx->d_cam, d_in.p, nb, d_out.p);
    LAUNCHED();
    CK(cudaMemcpyAsync(out, d_out.p, nb * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    return PNA_OK;
}

// ------------------------------------------------------------------------------------------------
// seam 3: encode -- implemented in encode_host.cuh on top of kernels_encode.cuh
#include "encode_host.cuh"
