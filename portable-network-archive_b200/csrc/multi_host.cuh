// multi_host.cuh -- a pna_ctx over several GPUs of one box (pna_cuda_init with n_devices > 1; included by abi.cu right after
// struct pna_plan).  Everything here works through the exports of pna_cuda.h on the per-device contexts and plans.
//
// Entries are independent units (own IV, own compressed stream, own chunks), so every batch call shards BY ENTRY: greedy
// longest-processing-time on stream bytes, one single-device context and one host thread per GPU, no peer traffic and no
// collective (SURVEY 8e; the reference's counterpart is the per-entry task fan-out of cli/src/command/extract.rs:868-1019).
// A multi-device plan is a list of ordinary single-device plans plus the index maps that put results back in caller order.
#pragma once
#include <thread>

namespace pna { namespace multi {

// LPT: heaviest entries first onto the least loaded device; each device keeps its entries in caller order
static std::vector<std::vector<uint32_t>> shard(const std::vector<uint64_t>& weight, size_t n_dev) {
    std::vector<uint32_t> order(weight.size());
    for (uint32_t i = 0; i < order.size(); i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return weight[a] > weight[b]; });
    std::vector<uint64_t> load(n_dev, 0);
    std::vector<std::vector<uint32_t>> part(n_dev);
    for (uint32_t i : order) {
        size_t best = 0;
        for (size_t d = 1; d < n_dev; d++) if (load[d] < load[best]) best = d;
        part[best].push_back(i);
        load[best] += weight[i] + 1;
    }
    for (auto& p : part) std::sort(p.begin(), p.end());
    return part;
}
// f(d) on one host thread per device; the first non-zero return code wins
template <class F>
static int for_devices(size_t n_dev, F&& f) {
    std::vector<int> rc(n_dev, PNA_OK);
    std::vector<std::thread> th;
    for (size_t d = 1; d < n_dev; d++) th.emplace_back([&, d]() { rc[d] = f(d); });
    rc[0] = f(0);
    for (auto& t : th) t.join();
    for (int r : rc) if (r != PNA_OK) return r;
    return PNA_OK;
}
static void carry_error(pna_ctx* root) {
    for (pna_ctx* c : root->devs) if (!c->err.empty()) { root->err = "device " + std::to_string(c->device) + ": " + c->err; return; }
}

// A per-entry export over the shards `part`: on device d's thread, call(d, idx, o, st) runs the single-device export on the
// caller entries idx = part[d] with o[k] = out[idx[k]]; on success every entry's length (pna_buf::len, or the length itself)
// and status go back to the caller's slots.
static uint64_t& length_of(pna_buf& b) { return b.len; }
static uint64_t& length_of(uint64_t& len) { return len; }
template <class T, class F>
static int per_entry(pna_ctx* root, const std::vector<std::vector<uint32_t>>& part, T* out, int32_t* status, F&& call) {
    const int rc = for_devices(part.size(), [&](size_t d) -> int {
        const auto& idx = part[d];
        if (idx.empty()) return PNA_OK;
        std::vector<T> o(idx.size());
        std::vector<int32_t> st(idx.size());
        for (size_t k = 0; k < idx.size(); k++) o[k] = out[idx[k]];
        const int r = call(d, idx, o.data(), st.data());
        if (r == PNA_OK) for (size_t k = 0; k < idx.size(); k++) { length_of(out[idx[k]]) = length_of(o[k]); status[idx[k]] = st[k]; }
        return r;
    });
    if (rc) carry_error(root);
    return rc;
}

static int crc32(pna_ctx* root, const pna_span* spans, uint32_t n, uint32_t* crc_out) {
    std::vector<uint64_t> w(n);
    for (uint32_t i = 0; i < n; i++) w[i] = spans[i].len;
    const auto part = shard(w, root->devs.size());
    const int rc = for_devices(root->devs.size(), [&](size_t d) -> int {
        const auto& idx = part[d];
        if (idx.empty()) return PNA_OK;
        std::vector<pna_span> s(idx.size());
        std::vector<uint32_t> c(idx.size());
        for (size_t k = 0; k < idx.size(); k++) s[k] = spans[idx[k]];
        const int r = pna_cuda_crc32(root->devs[d], s.data(), (uint32_t)s.size(), c.data());
        if (r == PNA_OK) for (size_t k = 0; k < idx.size(); k++) crc_out[idx[k]] = c[k];
        return r;
    });
    if (rc) carry_error(root);
    return rc;
}
static int crc32_image(pna_ctx* root, const uint8_t* image, const uint64_t* span_off, const uint64_t* span_len, uint32_t n, uint32_t* crc_out) {
    std::vector<pna_span> sp(n);
    for (uint32_t i = 0; i < n; i++) sp[i] = {image + span_off[i], span_len[i]};
    return crc32(root, sp.data(), n, crc_out);
}

// ---- decode
static std::vector<uint64_t> stream_bytes(const pna_decode_desc* descs, uint32_t n) {
    std::vector<uint64_t> w(n);
    for (uint32_t i = 0; i < n; i++) { uint64_t b = 0; for (uint32_t k = 0; k < descs[i].n_bodies; k++) b += descs[i].bodies[k].len; w[i] = b; }
    return w;
}
// one ordinary batch per device
static int decode_batch(pna_ctx* root, const pna_decode_desc* descs, uint32_t n, pna_buf* out, int32_t* status) {
    return per_entry(root, shard(stream_bytes(descs, n), root->devs.size()), out, status,
                     [&](size_t d, const std::vector<uint32_t>& idx, pna_buf* b, int32_t* st) {
        std::vector<pna_decode_desc> dd(idx.size());
        for (size_t k = 0; k < idx.size(); k++) dd[k] = descs[idx[k]];
        return pna_cuda_decode_batch(root->devs[d], dd.data(), (uint32_t)dd.size(), b, st);
    });
}

struct Plan {   // hangs off pna_plan::multi
    std::vector<pna_plan*> sub;                   // one per device (null: no entry landed there)
    std::vector<std::vector<uint32_t>> idx;       // sub[d] entry k == caller entry idx[d][k]
    std::vector<std::vector<uint32_t>> crc_idx;   // sub[d] CRC span k == caller span crc_idx[d][k]
    std::vector<uint32_t> where_dev, where_loc;   // caller entry -> (device, local index)
    std::vector<uint64_t> crc_count_bound;        // encode: pna_cuda_encode_crc_count of every caller entry
    Plan(const std::vector<uint64_t>& weight, size_t n_dev)
        : sub(n_dev, nullptr), idx(shard(weight, n_dev)), crc_idx(n_dev), where_dev(weight.size(), 0), where_loc(weight.size(), 0) {
        for (size_t d = 0; d < n_dev; d++) for (size_t k = 0; k < idx[d].size(); k++) { where_dev[idx[d][k]] = (uint32_t)d; where_loc[idx[d][k]] = (uint32_t)k; }
    }
};

// make(d) creates M->sub[d] on device d's thread; on failure the sub-plans made so far go, and M with them
template <class F>
static int plan_create(pna_ctx* root, Plan* M, int kind, uint32_t n, pna_plan** plan, F&& make) {
    const int rc = for_devices(M->sub.size(), make);
    if (rc) {
        carry_error(root);
        for (pna_plan* s : M->sub) if (s) pna_cuda_plan_destroy(s);
        delete M;
        return rc;
    }
    pna_plan* P = new pna_plan();
    P->ctx = root; P->kind = kind; P->n = n; P->multi = M;
    *plan = P;
    return PNA_OK;
}

static int decode_plan_create(pna_ctx* root, const pna_decode_desc* descs, uint32_t n, const CrcReq* crc, pna_plan** plan) {
    const size_t nd = root->devs.size();
    Plan* M = new Plan(stream_bytes(descs, n), nd);
    // a chunk travels with its entry; archive-level chunks (entry -1) are spread round-robin
    for (uint32_t c = 0, rr = 0; crc && c < crc->n; c++) M->crc_idx[crc->entry_of[c] >= 0 ? M->where_dev[crc->entry_of[c]] : (rr++ % nd)].push_back(c);
    return plan_create(root, M, 0, n, plan, [&](size_t d) -> int {
        const auto& idx = M->idx[d];
        const auto& cidx = M->crc_idx[d];
        if (idx.empty() && cidx.empty()) return PNA_OK;
        std::vector<pna_decode_desc> dd(idx.size());
        for (size_t k = 0; k < idx.size(); k++) dd[k] = descs[idx[k]];
        std::vector<pna_span> cs(cidx.size());
        std::vector<uint32_t> ce(cidx.size());
        std::vector<int32_t> co(cidx.size());
        for (size_t k = 0; k < cidx.size(); k++) {
            cs[k] = crc->spans[cidx[k]]; ce[k] = crc->expect[cidx[k]];
            co[k] = crc->entry_of[cidx[k]] >= 0 ? (int32_t)M->where_loc[crc->entry_of[cidx[k]]] : -1;
        }
        if (crc && crc->image) return pna_cuda_decode_plan_create_in_image(root->devs[d], dd.data(), (uint32_t)dd.size(), crc->image, crc->image_len, cs.data(),
                                                                           ce.data(), co.data(), (uint32_t)cs.size(), &M->sub[d]);
        if (crc) return pna_cuda_decode_plan_create_crc(root->devs[d], dd.data(), (uint32_t)dd.size(), cs.data(), ce.data(), co.data(),
                                                        (uint32_t)cs.size(), &M->sub[d]);
        return pna_cuda_decode_plan_create(root->devs[d], dd.data(), (uint32_t)dd.size(), &M->sub[d]);
    });
}

template <class F>
static int each_sub(pna_plan* P, F&& f) {
    Plan* M = P->multi;
    const int rc = for_devices(M->sub.size(), [&](size_t d) -> int { return M->sub[d] ? f(d, M->sub[d]) : PNA_OK; });
    if (rc) carry_error(P->ctx);
    return rc;
}
static int decode_plan_run(pna_plan* P) { return each_sub(P, [](size_t, pna_plan* s) { return pna_cuda_decode_plan_run(s); }); }
static int decode_plan_fetch(pna_plan* P, pna_buf* out, int32_t* status) {
    Plan* M = P->multi;
    return per_entry(P->ctx, M->idx, out, status, [&](size_t d, const std::vector<uint32_t>&, pna_buf* b, int32_t* st) {
        return pna_cuda_decode_plan_fetch(M->sub[d], b, st); });
}
static int decode_plan_lengths(pna_plan* P, uint64_t* out_len, int32_t* status) {
    Plan* M = P->multi;
    return per_entry(P->ctx, M->idx, out_len, status, [&](size_t d, const std::vector<uint32_t>&, uint64_t* l, int32_t* st) {
        return pna_cuda_decode_plan_lengths(M->sub[d], l, st); });
}
static int plan_crc_results(pna_plan* P, uint32_t* crc_out, uint32_t* n_broken) {
    Plan* M = P->multi;
    std::vector<uint32_t> broken(M->sub.size(), 0);
    const int rc = each_sub(P, [&](size_t d, pna_plan* s) -> int {
        const auto& cidx = M->crc_idx[d];
        std::vector<uint32_t> c(cidx.size());
        const int r = pna_cuda_plan_crc_results(s, crc_out ? c.data() : nullptr, &broken[d]);
        if (r == PNA_OK && crc_out) for (size_t k = 0; k < cidx.size(); k++) crc_out[cidx[k]] = c[k];
        return r;
    });
    if (n_broken) { *n_broken = 0; for (uint32_t b : broken) *n_broken += b; }
    return rc;
}
// the device plan that holds caller entry *entry, which becomes its index there (null: no such entry)
static pna_plan* route(pna_plan* P, uint32_t* entry) {
    Plan* M = P->multi;
    if (*entry >= P->n) return nullptr;
    pna_plan* sub = M->sub[M->where_dev[*entry]];
    *entry = M->where_loc[*entry];
    return sub;
}
static void sum_stats(pna_plan* P, uint64_t* a, uint64_t* b, uint64_t* c, bool counts) {
    uint64_t ta = 0, tb = 0, tc = 0;
    for (pna_plan* s : P->multi->sub) {
        if (!s) continue;
        uint64_t x = 0, y = 0, z = 0;
        if (counts) pna_cuda_plan_counts(s, &x, &y, &z); else pna_cuda_plan_stats(s, &x, &y, &z);
        ta += x; tb += y; tc += z;
    }
    if (a) *a = ta;
    if (b) *b = tb;
    if (c) *c = tc;
}
static int stage_ms(pna_plan* P, float* ms, uint32_t cap) {   // per stage: the slowest device
    int ns = 0;
    for (uint32_t i = 0; i < cap; i++) ms[i] = 0.f;
    for (pna_plan* s : P->multi->sub) {
        if (!s) continue;
        float t[32] = {0};
        const int k = pna_cuda_plan_stage_ms(s, t, 32);
        if (k < 0) return k;
        ns = std::max(ns, k);
        for (int i = 0; i < k && (uint32_t)i < cap; i++) ms[i] = std::max(ms[i], t[i]);
    }
    return ns;
}
static void plan_destroy(pna_plan* P) {
    Plan* M = P->multi;
    for (pna_plan* s : M->sub) if (s) pna_cuda_plan_destroy(s);
    delete M;
    P->multi = nullptr;
    delete P;
}

// ---- encode
static int encode_plan_create(pna_ctx* root, const pna_encode_desc* descs, uint32_t n, pna_plan** plan) {
    std::vector<uint64_t> w(n);
    for (uint32_t i = 0; i < n; i++) w[i] = descs[i].plain.len;
    Plan* M = new Plan(w, root->devs.size());
    M->crc_count_bound.resize(n);
    for (uint32_t i = 0; i < n; i++) M->crc_count_bound[i] = pna_cuda_encode_crc_count(&descs[i]);
    return plan_create(root, M, 1, n, plan, [&](size_t d) -> int {
        const auto& idx = M->idx[d];
        if (idx.empty()) return PNA_OK;
        std::vector<pna_encode_desc> dd(idx.size());
        for (size_t k = 0; k < idx.size(); k++) dd[k] = descs[idx[k]];
        return pna_cuda_encode_plan_create(root->devs[d], dd.data(), (uint32_t)dd.size(), &M->sub[d]);
    });
}
static int encode_plan_run(pna_plan* P) { return each_sub(P, [](size_t, pna_plan* s) { return pna_cuda_encode_plan_run(s); }); }
static int encode_plan_lengths(pna_plan* P, uint64_t* out_len, int32_t* status) {
    Plan* M = P->multi;
    return per_entry(P->ctx, M->idx, out_len, status, [&](size_t d, const std::vector<uint32_t>&, uint64_t* l, int32_t* st) {
        return pna_cuda_encode_plan_lengths(M->sub[d], l, st); });
}
static int encode_plan_fetch(pna_plan* P, pna_buf* out, uint32_t* fdat_crc_out, uint32_t* crc_count_out, int32_t* status) {
    Plan* M = P->multi;
    // per-device CRC lists, re-packed in caller order afterwards (the flat layout is consecutive per entry)
    std::vector<std::vector<uint32_t>> crcs(M->sub.size()), counts(M->sub.size());
    const int rc = each_sub(P, [&](size_t d, pna_plan* s) -> int {
        const auto& idx = M->idx[d];
        std::vector<pna_buf> b(idx.size());
        std::vector<int32_t> st(idx.size());
        uint64_t bound = 0;
        for (size_t k = 0; k < idx.size(); k++) { b[k] = out[idx[k]]; bound += M->crc_count_bound[idx[k]]; }
        crcs[d].resize(bound + 1); counts[d].resize(idx.size());
        const int r = pna_cuda_encode_plan_fetch(s, b.data(), crcs[d].data(), counts[d].data(), st.data());
        if (r == PNA_OK) for (size_t k = 0; k < idx.size(); k++) { out[idx[k]].len = b[k].len; status[idx[k]] = st[k]; }
        return r;
    });
    if (rc) return rc;
    std::vector<uint64_t> at(M->sub.size(), 0);   // read cursor per device: entries come back in local (= caller) order
    std::vector<std::vector<uint64_t>> start(M->sub.size());
    for (size_t d = 0; d < M->sub.size(); d++) {
        start[d].resize(M->idx[d].size());
        uint64_t pos = 0;
        for (size_t k = 0; k < M->idx[d].size(); k++) { start[d][k] = pos; pos += M->sub[d] ? counts[d][k] : 0; }
    }
    uint64_t pos = 0;
    for (uint32_t i = 0; i < P->n; i++) {
        const uint32_t d = M->where_dev[i], k = M->where_loc[i];
        const uint32_t c = M->sub[d] ? counts[d][k] : 0;
        if (crc_count_out) crc_count_out[i] = c;
        if (fdat_crc_out) for (uint32_t q = 0; q < c; q++) fdat_crc_out[pos + q] = crcs[d][start[d][k] + q];
        pos += c;
    }
    return PNA_OK;
}

}}  // namespace pna::multi
