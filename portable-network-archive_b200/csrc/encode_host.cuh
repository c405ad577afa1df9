// encode_host.cuh -- host side of seam 3 (included at the end of abi.cu): layout of the work arena, the launch
// sequence  match -> block writers -> layout -> encrypt -> FDAT CRC,  and the fetch.  The run is fully
// asynchronous: everything that depends on produced lengths is resolved on the device.
namespace pna { namespace enc {

struct EncodePlan {
    std::vector<EncEntry> h_entries;
    std::vector<SegRec> h_segs;
    KeyTable h_keys;
    std::vector<CipherTile> h_tiles[3];       // 0 none (gather), 1 aes-ctr, 2 camellia-ctr
    std::vector<uint32_t> h_cbc[2];           // aes, camellia
    std::vector<CrcTileSrc> h_crc_src;
    std::vector<uint32_t> h_crc_first;        // first tile of every body
    std::vector<uint32_t> crc_body_begin;     // per entry: first body
    std::vector<uint32_t> crc_body_size;      // per entry: max_chunk_size (bytes per body)
    uint64_t work_bytes = 0, out_bytes = 0, n_pieces = 0, seq_total = 0;
    DevArr<uint8_t> d_work, d_out;
    DevArr<EncEntry> d_entries, d_entries_init;
    DevArr<SegRec> d_segs;
    DevArr<Seq> d_seqs;
    DevArr<Segment> d_pieces;
    DevArr<DevKeys> d_keys;
    DevArr<CipherTile> d_tiles[3];
    DevArr<uint32_t> d_cbc[2], d_crc_first, d_crc_raw, d_crc_val;
    DevArr<CrcTileSrc> d_crc_src;
    DevArr<CrcTile> d_crc_tiles;
    DevArr<EncTables> d_tables;
    DevArr<uint8_t> d_stage;                  // coalesced transfers: many small adjacent host spans travel as one copy
    DevArr<CopyJob> d_stage_jobs;
    uint32_t fdat_init = 0;
    bool has_zstd = false, has_deflate = false, has_xz[4] = {false, false, false, false};   // which block writers the batch needs (xz: by literal-context setting)
    // GCM STREAM: segment / tile slots from the compressed-length bounds (AES slots first, then Camellia)
    std::vector<GcmSlot> h_gcm_slots;
    std::vector<gcm::GcmKeyRef> h_gcm_refs;
    DevArr<GcmSlot> d_gcm_slots;
    GcmDev gcm;
};
void destroy(EncodePlan* p) { delete p; }
// cipher kernels by slot: h_tiles / d_tiles (AES-CTR with AES_CTR_THREADS, one CTA per SM) and h_cbc / d_cbc
static const CipherKernel<decltype(&encrypt_tiles_kernel<0>)> ENCRYPT_TILES[3] = {
    {encrypt_tiles_kernel<0>, 0}, {encrypt_tiles_kernel<1>, AES_CTR_SMEM}, {encrypt_tiles_kernel<2>, CAM_SMEM}};
static const CipherKernel<decltype(&cbc_encrypt_kernel<1>)> CBC_ENCRYPT[2] = {{cbc_encrypt_kernel<1>, AES_SMEM}, {cbc_encrypt_kernel<2>, CAM_SMEM}};
bool init_attributes() {
    bool ok = cudaFuncSetAttribute(lz_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MATCH_SMEM_BYTES) == cudaSuccess &&
              cudaFuncSetAttribute(xz_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xz_enc_smem_bytes(xz::ENC_LC_MAX)) == cudaSuccess;
    for (const auto& k : ENCRYPT_TILES) ok = ok && k.opt_in();
    for (const auto& k : CBC_ENCRYPT) ok = ok && k.opt_in();
    return ok;
}
}}  // namespace pna::enc

using pna::enc::EncodePlan;
using pna::enc::EncEntry;

static uint64_t enc_nsegs(uint64_t len) { return (len + enc::SEG - 1) / enc::SEG; }
// upper bound of the compressed stream (before IV / padding): raw-block / stored-block fallbacks bound every segment
static uint64_t enc_comp_bound(uint8_t compression, uint64_t len) {
    if (compression == PNA_COMPRESSION_ZSTD) return len + 3 * enc_nsegs(len) + 9 + 6 * (enc_nsegs(len) / enc::FRAME_SEGS + 1);
    if (compression == PNA_COMPRESSION_DEFLATE) return len + 5 * enc_nsegs(len) + 8;
    if (compression == PNA_COMPRESSION_XZ) return len + 3 * enc_nsegs(len) + 24 + 48;   // uncompressed chunks + container
    return len;
}
static bool enc_is_gcm(const pna_encode_desc& d) { return d.encryption != 0 && d.cipher_mode == PNA_CIPHER_GCM; }
static uint32_t enc_gcm_seg_size(const pna_encode_desc& d) {   // 0: no / invalid header
    if (!d.stream_header) return 0;
    const uint8_t* h = d.stream_header;
    const uint32_t s = (uint32_t)h[39] << 24 | (uint32_t)h[40] << 16 | (uint32_t)h[41] << 8 | h[42];
    return s <= gcm::GCM_MAX_SEGMENT ? s : 0;
}
// stream prefix that the caller splits off as its own chunk(s): IV (CBC/CTR) or stream header (GCM)  builder.rs:62-69
static uint64_t enc_prefix_len(const pna_encode_desc& d) { return d.encryption ? (enc_is_gcm(d) ? gcm::GCM_HEADER_LEN : 16) : 0; }
extern "C" uint64_t pna_cuda_encode_bound(const pna_encode_desc* d) {
    if (!d) return 0;
    const uint64_t cb = enc_comp_bound(d->compression, d->plain.len);
    if (enc_is_gcm(*d)) {
        const uint32_t seg = enc_gcm_seg_size(*d);
        return gcm::GCM_HEADER_LEN + cb + (seg ? cb / seg + 1 : 1) * (uint64_t)gcm::GCM_TAG_LEN;
    }
    return cb + (d->encryption ? 32 : 0);
}
extern "C" uint64_t pna_cuda_encode_crc_count(const pna_encode_desc* d) {
    if (!d) return 0;
    const uint64_t cap = d->max_chunk_size ? d->max_chunk_size : 0xFFFFFFFFull;
    const uint64_t body = pna_cuda_encode_bound(d) - enc_prefix_len(*d);
    return (body + cap - 1) / cap + 1;
}

static int encode_plan_build(pna_ctx* ctx, const pna_encode_desc* descs, uint32_t n, pna_plan* P) {
    P->ctx = ctx; P->kind = 1; P->n = n;
    EncodePlan* E = new EncodePlan();
    P->enc = E;
    E->h_entries.resize(n);
    // work arena: [plain | literals (same layout) | per-segment tmp | per-entry header scratch]
    uint64_t plain_total = 0, nsegs_total = 0;
    for (uint32_t i = 0; i < n; i++) {
        const pna_encode_desc& d = descs[i];
        EncEntry& e = E->h_entries[i];
        memset(&e, 0, sizeof e);
        if (d.plain.len && !d.plain.ptr) return PNA_E_BAD_ARG;
        e.plain_off = plain_total; e.plain_len = d.plain.len;
        plain_total += align_up(d.plain.len, 16) + 16;
        e.compression = d.compression; e.encryption = d.encryption; e.cipher_mode = d.cipher_mode;
        e.effort = (uint8_t)enc::enc_effort(d.compression, d.level);
        if (d.compression == PNA_COMPRESSION_ZSTD) E->has_zstd = true;
        if (d.compression == PNA_COMPRESSION_DEFLATE) E->has_deflate = true;
        if (d.compression == PNA_COMPRESSION_XZ) E->has_xz[enc::xz_lc_for_effort(e.effort)] = true;
        memcpy(e.iv, d.iv, 16);
        e.key_idx = -1;
        e.status = entry_mode_status(d.compression, d.encryption, d.cipher_mode);
        if (e.status == ST_OK && enc_is_gcm(d) && enc_gcm_seg_size(d) == 0)
            e.status = ST_INVALID_INPUT;   // no stream header / segment size out of range (SegmentSize::new, aead.rs:83-88)
        if (e.status != ST_OK) continue;
        if (enc_is_gcm(d)) { e.gcm_seg_size = enc_gcm_seg_size(d); memcpy(e.gcm_hdr, d.stream_header, gcm::GCM_HEADER_LEN); }
        if (d.compression != PNA_COMPRESSION_NO) { e.seg_begin = (uint32_t)nsegs_total; e.n_segs = (uint32_t)enc_nsegs(d.plain.len); nsegs_total += e.n_segs; }
        if (d.encryption) e.key_idx = E->h_keys.index(ctx, d.encryption, d.key);
    }
    if (nsegs_total > 0xFFFFFFF0ull) return PNA_E_OOM;
    const uint64_t lit_base = align_up(plain_total, 256);
    const uint64_t tmp_base = lit_base + align_up(plain_total, 256);
    const uint64_t hdr_base = tmp_base + nsegs_total * enc::TMP_SEG;
    E->work_bytes = hdr_base + (uint64_t)n * xz::XZ_HDR_SCRATCH + 256;
    E->h_segs.resize(nsegs_total);
    uint64_t out_cur = 0, piece_cur = 0, crc_bodies = 0;
    E->crc_body_begin.resize(n); E->crc_body_size.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        EncEntry& e = E->h_entries[i];
        const pna_encode_desc& d = descs[i];
        e.hdr_off = hdr_base + (uint64_t)i * xz::XZ_HDR_SCRATCH;
        e.piece_begin = piece_cur;
        e.out_off = out_cur;
        E->crc_body_begin[i] = (uint32_t)crc_bodies;
        E->crc_body_size[i] = d.max_chunk_size ? d.max_chunk_size : 0xFFFFFFFFu;
        if (e.status != ST_OK) continue;
        for (uint32_t k = 0; k < e.n_segs; k++) {
            enc::SegRec& s = E->h_segs[e.seg_begin + k];
            memset(&s, 0, sizeof s);
            s.plain_off = e.plain_off + (uint64_t)k * enc::SEG;
            s.lit_off = lit_base + s.plain_off;
            s.tmp_off = tmp_base + (uint64_t)(e.seg_begin + k) * enc::TMP_SEG;
            s.seq_off = (uint64_t)(e.seg_begin + k) * enc::SEG_SEQ_MAX;
            s.len = (uint32_t)std::min<uint64_t>(enc::SEG, e.plain_len - (uint64_t)k * enc::SEG);
            s.entry = i;
            s.last = k + 1 == e.n_segs || (e.compression == PNA_COMPRESSION_ZSTD && (k + 1) % enc::FRAME_SEGS == 0);   // Last_Block of its frame
            s.adler = e.compression == PNA_COMPRESSION_DEFLATE;
            s.effort = e.effort;
        }
        piece_cur += 4 + 3 * (uint64_t)e.n_segs + e.n_segs / enc::FRAME_SEGS;
        const uint64_t bound = pna_cuda_encode_bound(&d);
        e.out_cap = bound;
        out_cur += align_up(bound, 16) + 16;
        // cipher work from the bound: CTR / none tiles, CBC list
        const uint64_t cb = enc_comp_bound(e.compression, e.plain_len);
        if (e.encryption && e.cipher_mode == PNA_CIPHER_CBC) E->h_cbc[e.encryption - 1].push_back(i);
        else if (e.encryption && e.cipher_mode == PNA_CIPHER_GCM) {
            // slots are laid out below (AES first, then Camellia)
        } else {
            std::vector<CipherTile>& tv = E->h_tiles[e.encryption];
            const uint64_t nb = (cb + 15) / 16;
            uint64_t b0 = 0;
            do {   // at least one tile per entry: it also writes the IV
                tv.push_back(CipherTile{i, (uint32_t)std::min<uint64_t>(CIPHER_TILE_BLOCKS, nb > b0 ? nb - b0 : 0), b0});
                b0 += CIPHER_TILE_BLOCKS;
            } while (b0 < nb);
        }
        // FDAT bodies after the IV (the IV is its own chunk, lib/src/entry/builder.rs:62-69)
        const uint64_t iv_len = enc_prefix_len(d), mcs = E->crc_body_size[i];
        const uint64_t nbody = (bound - iv_len + mcs - 1) / mcs + 1;
        for (uint64_t b = 0; b < nbody; b++) {
            E->h_crc_first.push_back((uint32_t)E->h_crc_src.size());
            const uint64_t lo = iv_len + b * mcs;
            uint64_t l = mcs;
            uint64_t o = lo;
            do {
                const uint32_t t = (uint32_t)std::min<uint64_t>(l, CRC_TILE);
                E->h_crc_src.push_back({o, t, i, (uint32_t)(crc_bodies + b)});
                o += t; l -= t;
            } while (l && o < bound + 16);
        }
        crc_bodies += nbody;
    }
    for (uint32_t pass = 1; pass <= 2; pass++) {
        for (uint32_t i = 0; i < n; i++) {
            EncEntry& e = E->h_entries[i];
            if (e.status != ST_OK || e.encryption != pass || e.cipher_mode != PNA_CIPHER_GCM) continue;
            const uint64_t cb = enc_comp_bound(e.compression, e.plain_len), S = e.gcm_seg_size;
            const uint64_t max_segs = cb / S + 1;
            const uint64_t tps = ((S + 15) / 16 + gcm::GCM_TILE_BLOCKS - 1) / gcm::GCM_TILE_BLOCKS;
            if (E->h_gcm_slots.size() + max_segs > 0x7FFFFFF0ull || (uint64_t)E->gcm.n_tiles + max_segs * tps > 0x7FFFFFF0ull) return PNA_E_OOM;
            e.gcm_slot_begin = (uint32_t)E->h_gcm_slots.size();
            e.gcm_tile_begin = E->gcm.n_tiles;
            e.gcm_tiles_per_seg = (uint32_t)tps;
            e.gcm_pow_idx = (uint32_t)E->h_gcm_refs.size();
            E->h_gcm_refs.push_back({e.key_idx, (uint32_t)e.encryption});
            for (uint64_t j = 0; j < max_segs; j++) E->h_gcm_slots.push_back({i, (uint32_t)j});
            E->gcm.n_tiles += (uint32_t)(max_segs * tps);
        }
        if (pass == 1) E->gcm.n_tiles_aes = E->gcm.n_tiles;
    }
    E->n_pieces = piece_cur;
    E->out_bytes = out_cur;
    E->seq_total = nsegs_total * enc::SEG_SEQ_MAX;
    if (crc_bodies > 0xFFFFFFF0ull || E->h_crc_src.size() > 0xFFFFFFF0ull) return PNA_E_OOM;
    // device arrays + upload; segments and keys get room even when there are none: kernels take their pointers
    CK(E->d_work.reserve(E->work_bytes)); CK(E->d_out.reserve(E->out_bytes + 256));
    CK(E->d_entries.reserve(n)); CK(E->d_entries_init.reserve(n));
    CK(E->d_segs.reserve(nsegs_total)); CK(E->d_seqs.reserve(E->seq_total + 8)); CK(E->d_pieces.reserve(piece_cur + 1));
    CK(E->d_keys.reserve(E->h_keys.keys.size()));
    {
        // Upload of the plaintext.  A cudaMemcpyAsync costs the host 5-10 us whatever its size, which is what a group of
        // thousands of small files is made of -- so runs of entries whose host spans are exactly adjacent (files packed into one
        // buffer, the common case) travel as ONE copy into a staging buffer and are scattered to their padded places by a kernel.
        constexpr uint64_t SMALL = 1 << 20, PIECE = 32 << 10;
        std::vector<CopyJob> jobs;
        struct Run { uint32_t lo, hi; uint64_t stage_off, bytes; };
        std::vector<Run> runs;
        uint64_t stage_bytes = 0;
        for (uint32_t i = 0; i < n;) {
            uint32_t j = i;
            uint64_t bytes = 0;
            auto ok = [&](uint32_t k) { return descs[k].plain.len && descs[k].plain.len < SMALL && E->h_entries[k].status == ST_OK; };
            if (ok(i)) {
                bytes = descs[i].plain.len;
                j = i + 1;
                while (j < n && ok(j) && descs[j - 1].plain.ptr + descs[j - 1].plain.len == descs[j].plain.ptr) { bytes += descs[j].plain.len; j++; }
            }
            if (j - i >= 4) { runs.push_back({i, j, stage_bytes, bytes}); stage_bytes += align_up(bytes, 256); i = j; continue; }
            const uint32_t end = j > i ? j : i + 1;
            for (uint32_t k = i; k < end; k++)
                if (descs[k].plain.len && E->h_entries[k].status == ST_OK)
                    CK(cudaMemcpyAsync(E->d_work.p + E->h_entries[k].plain_off, descs[k].plain.ptr, descs[k].plain.len, cudaMemcpyHostToDevice, ctx->stream));
            i = end;
        }
        if (!runs.empty()) {
            CK(E->d_stage.reserve(stage_bytes + 256));
            for (const Run& r : runs) {
                CK(cudaMemcpyAsync(E->d_stage.p + r.stage_off, descs[r.lo].plain.ptr, r.bytes, cudaMemcpyHostToDevice, ctx->stream));
                uint64_t at = r.stage_off;
                for (uint32_t k = r.lo; k < r.hi; k++) {
                    for (uint64_t o = 0; o < descs[k].plain.len; o += PIECE)
                        jobs.push_back({E->h_entries[k].plain_off + o, at + o, std::min<uint64_t>(PIECE, descs[k].plain.len - o)});
                    at += descs[k].plain.len;
                }
            }
            CK(E->d_stage_jobs.upload(jobs, ctx->stream));
            const uint32_t grid = std::min<uint32_t>(((uint32_t)jobs.size() + 7) / 8, (uint32_t)ctx->sm_count * 8);
            copy_jobs_kernel<<<grid, 256, 0, ctx->stream>>>(E->d_work.p, E->d_stage.p, E->d_stage_jobs.p, (uint32_t)jobs.size());
            LAUNCHED();
            CK(ctx->sync());   // `jobs` is a local; the staging buffer goes back to the cache
            E->d_stage.release();
        }
    }
    cudaStream_t s = ctx->stream;
    CK(E->d_entries_init.upload(E->h_entries, s)); CK(E->d_segs.upload(E->h_segs, s)); CK(E->d_keys.upload(E->h_keys.keys, s));
    static enc::EncTables h_tables;
    static std::once_flag h_tables_once;   // plans are built concurrently by the host layer's worker threads
    std::call_once(h_tables_once, []() { enc::make_enc_tables(&h_tables); });
    CK(E->d_tables.upload(&h_tables, 1, s));
    for (int v = 0; v < 3; v++) CK(E->d_tiles[v].upload(E->h_tiles[v], s));
    for (int v = 0; v < 2; v++) CK(E->d_cbc[v].upload(E->h_cbc[v], s));
    if (!E->h_gcm_slots.empty()) {
        GcmDev& G = E->gcm;
        G.n_segs = (uint32_t)E->h_gcm_slots.size(); G.n_keys = (uint32_t)E->h_gcm_refs.size();
        CK(E->d_gcm_slots.upload(E->h_gcm_slots, s)); CK(G.refs.upload(E->h_gcm_refs, s));
        CK(G.segs.reserve(G.n_segs)); CK(G.pows.reserve(G.n_keys)); CK(G.tiles.reserve(G.n_tiles + 1)); CK(G.partial.reserve(G.n_tiles + 1));
    }
    if (!E->h_crc_src.empty()) {
        CK(E->d_crc_src.upload(E->h_crc_src, s)); CK(E->d_crc_first.upload(E->h_crc_first, s));
        CK(E->d_crc_tiles.reserve(E->h_crc_src.size())); CK(E->d_crc_raw.reserve(E->h_crc_src.size())); CK(E->d_crc_val.reserve(E->h_crc_first.size()));
    }
    {   // register value after the chunk type: chunk CRC covers type || data (lib/src/format/chunk.rs:7-12)
        uint32_t c = 0xFFFFFFFFu;
        const uint8_t ty[4] = {'F', 'D', 'A', 'T'};
        for (int k = 0; k < 4; k++) { c ^= ty[k]; for (int b = 0; b < 8; b++) c = (c >> 1) ^ (CRC_POLY & (0u - (c & 1u))); }
        E->fdat_init = c;
    }
    CK(ctx->sync());   // the borrowed plaintext may go away after this call
    for (uint32_t i = 0; i < n; i++) P->plain_bytes += descs[i].plain.len;
    return PNA_OK;
}

static int encode_launch_all(pna_plan* P) {
    pna_ctx* ctx = P->ctx;
    EncodePlan* E = P->enc;
    const uint64_t l0 = ctx->launches;
    const uint32_t n = P->n, nsegs = (uint32_t)E->h_segs.size();
    int rc = lease_stage_events(P);
    if (rc) return rc;
    CK(cudaMemcpyAsync(E->d_entries.p, E->d_entries_init.p, n * sizeof(EncEntry), cudaMemcpyDeviceToDevice, ctx->stream));
    STAGE(0);
    if (nsegs) {
        enc::lz_match_kernel<<<(nsegs + enc::ENC_WARPS - 1) / enc::ENC_WARPS, 32 * enc::ENC_WARPS, enc::MATCH_SMEM_BYTES, ctx->stream>>>(
            E->d_work.p, E->d_work.p, E->d_segs.p, nsegs, E->d_seqs.p);
        LAUNCHED();
        STAGE(1);
        const uint32_t bgrid = (nsegs + enc::ENC_BLOCK_THREADS - 1) / enc::ENC_BLOCK_THREADS;
        if (E->has_zstd) {
            enc::enc_block_kernel<2><<<bgrid, enc::ENC_BLOCK_THREADS, 0, ctx->stream>>>(E->d_work.p, E->d_segs.p, nsegs, E->d_seqs.p, E->d_tables.p, E->d_entries.p);
            LAUNCHED();
        }
        if (E->has_deflate) {
            enc::enc_block_kernel<1><<<bgrid, enc::ENC_BLOCK_THREADS, 0, ctx->stream>>>(E->d_work.p, E->d_segs.p, nsegs, E->d_seqs.p, E->d_tables.p, E->d_entries.p);
            LAUNCHED();
        }
        for (uint32_t lc = 0; lc < 4; lc++) {
            if (!E->has_xz[lc]) continue;
            enc::xz_encode_kernel<<<nsegs, 32, enc::xz_enc_smem_bytes(lc), ctx->stream>>>(E->d_work.p, E->d_segs.p, nsegs, E->d_seqs.p, E->d_entries.p, lc);
            LAUNCHED();
        }
    }
    else STAGE(1);
    STAGE(2);
    enc::enc_layout_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(E->d_work.p, E->d_segs.p, E->d_entries.p, n, E->d_pieces.p);
    LAUNCHED();
    STAGE(3);
    for (int v = 0; v < 3; v++) {
        const uint32_t nt = (uint32_t)E->h_tiles[v].size();
        if (!nt) continue;
        const auto encrypt_tiles = enc::ENCRYPT_TILES[v].fn;
        encrypt_tiles<<<std::min<uint32_t>(nt, (uint32_t)ctx->sm_count * (v == 1 ? 1 : 6)), v == 1 ? AES_CTR_THREADS : 256, enc::ENCRYPT_TILES[v].smem,
                        ctx->stream>>>(E->d_work.p, E->d_pieces.p, E->d_entries.p, E->d_tiles[v].p, nt, E->d_keys.p, ctx->d_aes, ctx->d_cam, E->d_out.p);
        LAUNCHED();
    }
    for (int v = 0; v < 2; v++) {
        const uint32_t nc = (uint32_t)E->h_cbc[v].size();
        if (!nc) continue;
        const auto cbc_encrypt = enc::CBC_ENCRYPT[v].fn;
        cbc_encrypt<<<(nc + 63) / 64, 64, enc::CBC_ENCRYPT[v].smem, ctx->stream>>>(E->d_work.p, E->d_pieces.p, E->d_entries.p, E->d_cbc[v].p, nc, E->d_keys.p,
                                                                                 ctx->d_aes, ctx->d_cam, E->d_out.p);
        LAUNCHED();
    }
    if (const uint32_t ns = E->gcm.n_segs) {
        enc::gcm_enc_slots_kernel<<<(ns + 127) / 128, 128, 0, ctx->stream>>>(E->d_gcm_slots.p, ns, E->d_entries.p, E->gcm.segs.p, E->gcm.tiles.p, E->d_out.p);
        LAUNCHED();
        if ((rc = launch_gcm<false>(ctx, E->gcm, E->d_work.p, E->d_pieces.p, E->d_out.p, nullptr, E->d_keys.p))) return rc;
    }
    STAGE(4);
    const uint32_t nt = (uint32_t)E->h_crc_src.size();
    if (nt) {
        enc::crc_clip_kernel<<<(nt + 127) / 128, 128, 0, ctx->stream>>>(E->d_crc_src.p, nt, E->d_entries.p, E->d_crc_tiles.p);
        LAUNCHED();
        if ((rc = launch_chunk_crc(ctx, E->d_out.p, E->d_crc_tiles.p, nt, E->d_crc_raw.p, E->d_crc_first.p, (uint32_t)E->h_crc_first.size(),
                                   E->d_crc_val.p, E->fdat_init)))
            return rc;
    }
    STAGE(5);
    for (int k = 6; k <= PNA_N_STAGES; k++) STAGE(k);
    P->ev_recorded = true;
    P->launches_per_run = ctx->launches - l0;
    P->prepared = true;
    return PNA_OK;
}
extern "C" const char* pna_cuda_encode_stage_name(uint32_t i) {
    static const char* const names[5] = {"lz_match", "block_write", "layout", "cipher", "crc"};
    return i < 5 ? names[i] : "";
}

extern "C" int pna_cuda_encode_plan_create(pna_ctx* ctx, const pna_encode_desc* descs, uint32_t n, pna_plan** plan) {
    if (!ctx || !plan || (!descs && n)) return PNA_E_BAD_ARG;
    *plan = nullptr;
    if (!ctx->devs.empty()) return multi::encode_plan_create(ctx, descs, n, plan);
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    pna_plan* P = new pna_plan();
    int rc = n ? encode_plan_build(ctx, descs, n, P) : (P->ctx = ctx, P->kind = 1, PNA_OK);
    if (rc) { delete P; return rc; }
    *plan = P;
    return PNA_OK;
}
extern "C" int pna_cuda_encode_plan_run(pna_plan* P) {
    if (!P || P->kind != 1) return PNA_E_BAD_ARG;
    if (P->multi) return multi::encode_plan_run(P);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    return encode_launch_all(P);
}
extern "C" int pna_cuda_encode_plan_lengths(pna_plan* P, uint64_t* out_len, int32_t* status) {
    if (!P || P->kind != 1 || ((!out_len || !status) && P->n)) return PNA_E_BAD_ARG;
    if (P->multi) return multi::encode_plan_lengths(P, out_len, status);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    if (!P->prepared) return PNA_E_BAD_ARG;
    std::vector<EncEntry> dev(P->n);
    CK(cudaMemcpyAsync(dev.data(), P->enc->d_entries.p, P->n * sizeof(EncEntry), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    for (uint32_t i = 0; i < P->n; i++) { status[i] = dev[i].status; out_len[i] = dev[i].status == ST_OK ? dev[i].out_len : 0; }
    return PNA_OK;
}
static int encode_plan_fetch_impl(pna_plan* P, pna_buf* out, uint32_t* fdat_crc_out, uint32_t* crc_count_out, int32_t* status, uint8_t* region,
                                  uint64_t region_len);
extern "C" int pna_cuda_encode_plan_fetch(pna_plan* P, pna_buf* out, uint32_t* fdat_crc_out, uint32_t* crc_count_out, int32_t* status) {
    return encode_plan_fetch_impl(P, out, fdat_crc_out, crc_count_out, status, nullptr, 0);
}
extern "C" int pna_cuda_encode_plan_fetch_region(pna_plan* P, pna_buf* out, uint8_t* region, uint64_t region_len, uint32_t* fdat_crc_out,
                                                 uint32_t* crc_count_out, int32_t* status) {
    if (!region && region_len) return PNA_E_BAD_ARG;
    return encode_plan_fetch_impl(P, out, fdat_crc_out, crc_count_out, status, region, region_len);
}
static int encode_plan_fetch_impl(pna_plan* P, pna_buf* out, uint32_t* fdat_crc_out, uint32_t* crc_count_out, int32_t* status, uint8_t* region,
                                  uint64_t region_len) {
    if (!P || P->kind != 1 || ((!out || !status) && P->n)) return PNA_E_BAD_ARG;
    if (P->multi) return multi::encode_plan_fetch(P, out, fdat_crc_out, crc_count_out, status);
    pna_ctx* ctx = P->ctx;
    std::lock_guard<std::mutex> g(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    if (P->n == 0) return PNA_OK;
    if (!P->prepared) return PNA_E_BAD_ARG;
    EncodePlan* E = P->enc;
    std::vector<EncEntry> dev(P->n);
    std::vector<uint32_t> crcs(E->h_crc_first.size());
    CK(cudaMemcpyAsync(dev.data(), E->d_entries.p, P->n * sizeof(EncEntry), cudaMemcpyDeviceToHost, ctx->stream));
    if (fdat_crc_out && !crcs.empty())
        CK(cudaMemcpyAsync(crcs.data(), E->d_crc_val.p, crcs.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx->sync());
    uint64_t stream_bytes = 0, crc_pos = 0;
    // The caller owns `region` entirely and every stream lands inside it: when the streams are many and close together (a
    // group of small files on their way into an archive, frames between them), the device lays them out as they will lie
    // in the region and ONE copy brings the whole span down; what lies between the streams is unspecified afterwards.
    bool staged = false;
    if (region && P->n >= 16) {
        const uint8_t* lo = nullptr; const uint8_t* hi = nullptr;
        uint64_t total = 0;
        bool fits = true;
        for (uint32_t i = 0; i < P->n; i++) {
            const EncEntry& e = dev[i];
            if (e.status != ST_OK || e.out_len == 0) continue;
            if (e.out_len > out[i].cap) continue;   // reported below as NOSPACE, not copied
            if (out[i].ptr < region || out[i].ptr + e.out_len > region + region_len) { fits = false; break; }
            if (!lo || out[i].ptr < lo) lo = out[i].ptr;
            if (!hi || out[i].ptr + e.out_len > hi) hi = out[i].ptr + e.out_len;
            total += e.out_len;
        }
        const uint64_t span = lo ? (uint64_t)(hi - lo) : 0;
        if (fits && lo && total / P->n < (1u << 20) && span <= total + total / 4 + 4096) {
            constexpr uint64_t PIECE = 32 << 10;
            std::vector<CopyJob> jobs;
            for (uint32_t i = 0; i < P->n; i++) {
                const EncEntry& e = dev[i];
                if (e.status != ST_OK || e.out_len == 0 || e.out_len > out[i].cap) continue;
                for (uint64_t o = 0; o < e.out_len; o += PIECE)
                    jobs.push_back({(uint64_t)(out[i].ptr - lo) + o, e.out_off + o, std::min<uint64_t>(PIECE, e.out_len - o)});
            }
            CK(E->d_stage.reserve(span + 256)); CK(E->d_stage_jobs.upload(jobs, ctx->stream));
            const uint32_t grid = std::min<uint32_t>(((uint32_t)jobs.size() + 7) / 8, (uint32_t)ctx->sm_count * 8);
            copy_jobs_kernel<<<grid, 256, 0, ctx->stream>>>(E->d_stage.p, E->d_out.p, E->d_stage_jobs.p, (uint32_t)jobs.size());
            LAUNCHED();
            CK(cudaMemcpyAsync(const_cast<uint8_t*>(lo), E->d_stage.p, span, cudaMemcpyDeviceToHost, ctx->stream));
            CK(ctx->sync());   // `jobs` is a local
            staged = true;
        }
    }
    for (uint32_t i = 0; i < P->n; i++) {
        const EncEntry& e = dev[i];
        int32_t st = e.status;
        uint64_t len = st == ST_OK ? e.out_len : 0;
        if (st == ST_OK && len > out[i].cap) st = ST_NOSPACE;
        out[i].len = (st == ST_OK || st == ST_NOSPACE) ? e.out_len : 0;
        status[i] = st;
        uint32_t nbody = 0;
        if (st == ST_OK) {
            if (len && !staged) CK(cudaMemcpyAsync(out[i].ptr, E->d_out.p + e.out_off, len, cudaMemcpyDeviceToHost, ctx->stream));
            stream_bytes += len;
            const uint64_t iv_len = e.encryption ? (e.cipher_mode == PNA_CIPHER_GCM ? gcm::GCM_HEADER_LEN : 16) : 0, mcs = E->crc_body_size[i];
            nbody = (uint32_t)((len - iv_len + mcs - 1) / mcs);
            if (fdat_crc_out)
                for (uint32_t b = 0; b < nbody; b++) fdat_crc_out[crc_pos + b] = crcs[E->crc_body_begin[i] + b];
        }
        if (crc_count_out) crc_count_out[i] = nbody;
        crc_pos += nbody;
    }
    P->stream_bytes = stream_bytes;
    CK(ctx->sync());
    return PNA_OK;
}
extern "C" int pna_cuda_encode_batch(pna_ctx* ctx, const pna_encode_desc* descs, uint32_t n, pna_buf* out, uint32_t* fdat_crc_out,
                                     uint32_t* crc_count_out, int32_t* status) {
    if (!ctx || ((!descs || !out || !status) && n)) return PNA_E_BAD_ARG;
    if (n == 0) return PNA_OK;
    pna_plan* P = nullptr;
    int rc = pna_cuda_encode_plan_create(ctx, descs, n, &P);
    if (rc) return rc;
    rc = pna_cuda_encode_plan_run(P);
    if (rc == PNA_OK) rc = pna_cuda_encode_plan_fetch(P, out, fdat_crc_out, crc_count_out, status);
    pna_cuda_plan_destroy(P);
    return rc;
}
