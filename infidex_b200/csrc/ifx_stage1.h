// infidex_b200 -- Stage 1 on device: query term resolution, LD1 expansion, tiered candidate selection,
// BM25+ with MaxScore over 4096-candidate chunks, exact emulation of the reference's pruning heap, top-K.
//
// What each routine replaces in the reference (src/Infidex/...):
//   prepare_query   Scoring/QueryAnalyzer.cs:10-54, Tokenization/Tokenizer.cs:144-200, Indexing/VectorModel.cs:376-563
//   expand_fuzzy    Indexing/Fst/FstIndex.cs:202-352 (MatchWithinEditDistance1), Indexing/VectorModel.cs:643-743
//   stage1_query    Scoring/TieredCandidateSelector.cs:53-532, Indexing/Bm25Scorer.cs:56-445,654-670
// Written against ifx::Ctx (one CTA on the GPU).
#pragma once
#include "ifx_base.h"

namespace ifx {

IFX_FN bool is_delim(const DevIndex& ix, uint16_t c) { return ix.cflags[c] & 4; }
IFX_FN bool is_space(const DevIndex& ix, uint16_t c) { return ix.cflags[c] & 2; }

IFX_FN int cmp_ordinal(const uint16_t* a, int na, const uint16_t* b, int nb) {   // string.CompareOrdinal
    int n = na < nb ? na : nb;
    for (int i = 0; i < n; i++) if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
    return na == nb ? 0 : (na < nb ? -1 : 1);
}

IFX_FN float max_term_score(float idf, float avgdl) {   // VectorModel.cs:523-531
    const float maxTf = 255.f, k1 = 1.2f, b = 0.75f, delta = 1.0f;
    float minDlNorm = 1.f - b + b * (1.f / avgdl);
    float core = (maxTf * (k1 + 1.f)) / (maxTf + k1 * minDlNorm);
    return idf * (core + delta);
}

// ---------------------------------------------------------------------------------------------------------------
// prepare_query: one thread per query.
IFX_FN void prepare_query(const DevIndex& ix, const uint16_t* text, int len, int depth, int max_results, int enable_cov,
                          int filter_id, int enable_facets, QueryPlan& p, FuzzyItem* items, int items_cap, BatchCounters* bc, int qi) {
    p.status = 0; p.n_terms = 0; p.n_fuzzy = 0; p.qlen = 0; p.tlen = 0; p.depth = depth; p.max_results = max_results;
    p.enable_coverage = enable_cov; p.filter_id = filter_id; p.enable_facets = enable_facets; p.short_skip_coverage = 0; p.is_short3 = 0; p.short_kind = 0; p.short_no_cov = 0;
    if (len > MAX_QLEN || depth > MAX_K || depth < 1) { p.status = 4; return; }
    bool blank = true;
    for (int i = 0; i < len; i++) { p.qtext[i] = text[i]; if (!is_space(ix, text[i])) blank = false; }
    p.qlen = len;
    if (blank) { p.status = 8; return; }
    // QueryAnalyzer.Analyze
    int n_words = 0, n_long = 0, n_short = 0, tl = 0;
    for (int i = 0; i < len;) {
        while (i < len && is_delim(ix, text[i])) i++;
        if (i >= len) break;
        int b = i; while (i < len && !is_delim(ix, text[i])) i++;
        n_words++;
        if (i - b > MAX_TOKLEN) p.status |= 4;      // the coverage kernel's Levenshtein row (ifx_cov.h lev) cannot hold this word: flagged, never silently unmatched
        if (i - b >= 3) { if (n_long > 0) p.ttext[tl++] = u' '; for (int k = b; k < i; k++) p.ttext[tl++] = text[k]; n_long++; } else n_short++;
    }
    bool can_ngrams = n_words == 0 ? len >= 3 : n_long > 0;
    if (!can_ngrams) {      // no word of >= 3 characters: ShortQueryProcessor / ShortQueryResolver (SearchPipeline.cs:222-262), scored by the launches of ifx_short.h
        if (ix.prefix_gcard || ix.key_first) { p.status |= 2; return; }      // a doc-id-range shard, or documents sharing a DocumentKey (the reference accumulates short-query scores per KEY): that combination is not built -- flagged (IFX_Q_UNSUPPORTED_OP), never answered partially
        p.short_kind = len == 1 ? 1 : 2; p.tlen = 0;
        bool short3 = len <= 3; for (int i = 0; i < len; i++) if (is_delim(ix, text[i])) short3 = false;
        p.is_short3 = short3; int64_t pc = -1;
        if (short3) { int k = dict_lookup(ix.prefix.keys, text, len); pc = k < 0 ? 0 : (ix.prefix_gcard ? (int64_t)ix.prefix_gcard[k] : ix.prefix.row_ptr[k + 1] - ix.prefix.row_ptr[k]); if (pc > 500) p.short_skip_coverage = 1; }
        p.short_no_cov = !(short3 && pc > 0 && pc <= 500);      // allowShortQueryCoverage (SearchPipeline.cs:133-137)
        return;
    }
    bool mixed = n_short > 0 && n_long > 0;
    if (!mixed) { tl = len; for (int i = 0; i < len; i++) p.ttext[i] = text[i]; }
    p.tlen = tl;
    // SearchPipeline.cs:110-142 short (<= 3 chars, no delimiter) query rules
    bool short3 = len <= 3; for (int i = 0; i < len; i++) if (is_delim(ix, text[i])) short3 = false;
    p.is_short3 = short3;
    if (short3) { int k = dict_lookup(ix.prefix.keys, text, len); if (k >= 0 && (ix.prefix_gcard ? (int64_t)ix.prefix_gcard[k] : ix.prefix.row_ptr[k + 1] - ix.prefix.row_ptr[k]) > 500) p.short_skip_coverage = 1; }
    // tokens: words (len >= 3) then padded 3-grams (Tokenizer.EnumerateShinglesForSearch), first 128 kept
    uint16_t padded[MAX_QLEN + 2]; padded[0] = PAD; padded[1] = PAD; for (int i = 0; i < tl; i++) padded[2 + i] = p.ttext[i];
    struct Raw { int32_t id; uint16_t off, len; };
    Raw raw[MAX_RAW_TOKENS]; int nr = 0;
    for (int i = 0; i < tl && nr < MAX_RAW_TOKENS;) {
        while (i < tl && is_delim(ix, p.ttext[i])) i++;
        if (i >= tl) break;
        int b = i; while (i < tl && !is_delim(ix, p.ttext[i])) i++;
        if (i - b >= 3) { raw[nr].off = (uint16_t)(b + 2); raw[nr].len = (uint16_t)(i - b); nr++; }
    }
    for (int k = 0; k + 3 <= tl + 2 && nr < MAX_RAW_TOKENS; k++) {
        if (padded[k] == PAD && padded[k + 1] == PAD && padded[k + 2] == PAD) continue;
        raw[nr].off = (uint16_t)k; raw[nr].len = 3; nr++;
    }
    for (int i = 0; i < nr; i++) raw[i].id = dict_lookup(ix.terms, padded + raw[i].off, raw[i].len);
    // RawToken.CompareTo: (TermId, ordinal text); equal elements are interchangeable so any sort gives the same sequence
    for (int i = 1; i < nr; i++) {
        Raw t = raw[i]; int j = i - 1;
        while (j >= 0) {
            int c = raw[j].id != t.id ? (raw[j].id < t.id ? -1 : 1) : (t.id >= 0 ? 0 : cmp_ordinal(padded + raw[j].off, raw[j].len, padded + t.off, t.len));
            if (c <= 0) break;
            raw[j + 1] = raw[j]; j--;
        }
        raw[j + 1] = t;
    }
    float avgdl = ix.avgdl > 0.f ? ix.avgdl : 1.f;
    int nt = 0;
    for (int i = 0; i < nr; i++) {
        if (i > 0 && raw[i].id == raw[i - 1].id && (raw[i].id >= 0 || cmp_ordinal(padded + raw[i].off, raw[i].len, padded + raw[i - 1].off, raw[i - 1].len) == 0)) continue;
        if (raw[i].id >= 0) {
            int df = ix.df[raw[i].id];
            if (df <= 0 || df > ix.stop_term_limit) continue;
            QTerm& t = p.terms[nt++];
            t.term_id = raw[i].id; t.df = df; t.list_off = ix.row_ptr[raw[i].id]; t.list_len = (int32_t)(ix.row_ptr[raw[i].id + 1] - ix.row_ptr[raw[i].id]);
            t.idf = compute_idf(ix, df); t.max_score = max_term_score(t.idf, avgdl);
        } else if (raw[i].len >= 4) {
            if (p.n_fuzzy >= MAX_FUZZY || raw[i].len > 64) { p.status |= 4; continue; }
            int slot = atomic_add(&bc->n_fuzzy_items, 1);
            if (slot >= items_cap) { p.status |= 4; continue; }
            QTerm& t = p.terms[nt]; t.term_id = -1; t.df = 0; t.list_off = 0; t.list_len = 0; t.idf = 0.f; t.max_score = 0.f;
            FuzzyReq& f = p.fuzzy[p.n_fuzzy++]; f.off = (uint16_t)(raw[i].off - 2); f.len = raw[i].len; f.term_slot = nt;
            items[slot].query = qi; items[slot].slot = p.n_fuzzy - 1;
            nt++;
        }
    }
    p.n_terms = nt;
}

// ---------------------------------------------------------------------------------------------------------------
// block primitives
struct ScanTmp { int w[33]; };

IFX_FN int block_excl_scan(const Ctx& c, int v, ScanTmp& tmp, int& total) {
#ifdef IFX_EMU
    (void)c; (void)tmp; total = v; return 0;
#else
    int incl = v;
    for (int d = 1; d < 32; d <<= 1) { int o = __shfl_up_sync(0xffffffffu, incl, d); if (c.lane() >= d) incl += o; }
    if (c.lane() == 31) tmp.w[c.warp()] = incl;
    c.sync();
    int base = 0, tot = 0, nw = c.nwarps();
    for (int i = 0; i < nw; i++) { int x = tmp.w[i]; if (i < c.warp()) base += x; tot += x; }
    total = tot;
    c.sync();
    return base + incl - v;
#endif
}
// single-barrier variant: callers alternate between two ScanTmp buffers (the barrier of the next call protects reuse)
IFX_FN int block_excl_scan_1b(const Ctx& c, int v, ScanTmp& tmp, int& total) {
#ifdef IFX_EMU
    (void)c; (void)tmp; total = v; return 0;
#else
    int incl = v;
    for (int d = 1; d < 32; d <<= 1) { int o = __shfl_up_sync(0xffffffffu, incl, d); if (c.lane() >= d) incl += o; }
    if (c.lane() == 31) tmp.w[c.warp()] = incl;
    c.sync();
    int base = 0, tot = 0, nw = c.nwarps();
    for (int i = 0; i < nw; i++) { int x = tmp.w[i]; if (i < c.warp()) base += x; tot += x; }
    total = tot;
    return base + incl - v;
#endif
}
IFX_FN int block_sum(const Ctx& c, int v, ScanTmp& tmp) { int t; block_excl_scan(c, v, tmp, t); return t; }

IFX_FN int64_t lower_bound_i32(const int32_t* a, int64_t lo, int64_t hi, int32_t target) {   // first index in [lo,hi) with a[i] >= target
    while (lo < hi) { int64_t mid = lo + ((hi - lo) >> 1); if (a[mid] < target) lo = mid + 1; else hi = mid; }
    return lo;
}

// lower bound executed by one full warp: 32-way splits instead of binary halving (log32 n dependent loads).
// Every lane of the calling warp must participate; the result is uniform across the warp.
IFX_FN int64_t warp_lower_bound(const Ctx& c, const int32_t* a, int64_t lo, int64_t hi, int32_t target) {
#ifdef IFX_EMU
    (void)c; return lower_bound_i32(a, lo, hi, target);
#else
    while (hi - lo > 32) {   // invariant: a[x] < target for x < lo, a[x] >= target for x >= hi
        int64_t step = (hi - lo + 31) / 32; int64_t p = lo + (int64_t)(c.lane() + 1) * step - 1; if (p > hi - 1) p = hi - 1;
        unsigned m = __ballot_sync(0xffffffffu, a[p] < target); int k = __popc(m);          // probes are monotone: lanes [0,k) see "less"
        int64_t pk = lo + (int64_t)(k + 1) * step - 1; if (pk > hi - 1) pk = hi - 1;          // first probe that is >= target (k < 32)
        int64_t pk1 = lo + (int64_t)k * step - 1; if (pk1 > hi - 1) pk1 = hi - 1;            // last probe that is < target (k > 0)
        if (k == 32) { lo = hi; break; }
        if (k > 0) lo = pk1 + 1;
        hi = pk;
    }
    int64_t i = lo + c.lane(); bool less = i < hi && a[i] < target;
    unsigned m = __ballot_sync(0xffffffffu, less);
    return lo + __popc(m);
#endif
}

// per-CTA global workspace
struct S1Workspace {
    unsigned* bits;        // candidate bitset over the shard's docs (all zero between uses)
    unsigned* bits2;       // membership bitset of the running AND-tier intersection (all zero between uses)
    int32_t* cand;         // sorted candidate ids
    int32_t* buf_a; int32_t* buf_b;   // AND-tier ping-pong arrays
    unsigned long long* surv_g;       // [CHUNK] flush survivors of one chunk when they exceed the shared staging buffer
    int32_t* lrange;       // [MAX_TERMS][n_cont + 1] per streamed list of the tf lookups: index of its first posting in container c
    int32_t* cstart;       // [n_cont + 1] candidates before container c
    int32_t* cfirst;       // [n_cont + 1] chunks before container c
    int32_t* ctab;         // [n_cont] packed S1Cont records (16 bytes each) for the tf lookups
    int64_t cand_cap, buf_cap;
};

struct TermS {             // term as seen by the scorer
    const int32_t* docs; const uint8_t* tf; const int32_t* skip; const unsigned* bm; const int32_t* bmr; int32_t len; int32_t df; float idf, max_score, suffix_after; int32_t term_id; int64_t cursor, s0, s1;
};

constexpr int S1_TILE = 6;

constexpr int SURV_CAP = 512;
constexpr int QH_SIZE = 256;
constexpr int SMALL_CHUNK = 512;                               // chunks up to this size are scored by a single warp, without block barriers
constexpr int SMALL_TERMS = S1_TILE * CHUNK / SMALL_CHUNK;      // ... when all their terms fit the tile buffer re-cut as [term][SMALL_CHUNK]
IFX_FN unsigned qh_hash(int32_t term_id) { return ((unsigned)term_id * 2654435761u) >> 24; }     // 8 bits = QH_SIZE
// shared memory of the selection / tf-lookup kernel (small: four 256-thread CTAs per SM)
struct S1SelShared {
    TermS terms[MAX_TERMS];
    int order[MAX_TERMS];
    int n_terms;
    int32_t qh_key[QH_SIZE]; uint8_t qh_slot[QH_SIZE];   // term id -> slot in `terms` (open addressing; terms with idf > 0 only), for the forward-index lookups
    uint8_t dirty[MAX_CONTAINERS];          // containers of the global bitset touched by the current set operation (all zero between uses)
    ScanTmp scan; ScanTmp scan2[2];
    int bcast[8]; long long bcast64[4];
    unsigned long long streamed_mask[2];   // terms whose list the selector streamed in full (roofline accounting)
};
// ... plus what the block-wide scorer and the LD1 expansion need
struct S1Shared : S1SelShared {
    alignas(16) float score[CHUNK];
    alignas(16) uint8_t tfm[S1_TILE][CHUNK];   // one tile of term rows of the current chunk
    int32_t cand_s[CHUNK]; alignas(16) float nv_s[CHUNK];   // per-slot length norm of the vector form (the scalar form is needed for < 8 matches per term and chunk: recomputed)
    unsigned ballots[2][CHUNK / Ctx::WS + 8]; int bprefix[CHUNK / Ctx::WS + 8];
    int heap_size; float thr;
    // .NET PriorityQueue nodes, stored with a +3 shift so the four children of node i (4i+1..4i+4) form one aligned 16-byte group; slots beyond
    // the current size hold +huge sentinels
    alignas(16) float heap_pr[MAX_K + 8]; int32_t heap_doc[MAX_K + 8];   // split so that one 16-byte load fetches the four child priorities
    unsigned long long surv[SURV_CAP];     // (doc, score) of the last chunk's flush survivors, drained into the heap while the next chunk is staged
    alignas(16) unsigned scan3[32][4];   // packed per-warp totals of the batched rank scan
    unsigned long long peq[128];           // Myers pattern masks of the word being expanded (ASCII fast path)
};

// Stream a sorted id list and hand it to `put(word, mask)` as per-32-bit-word masks (word = id >> 5).
// Long lists: every thread takes runs of 8 consecutive ids (two 16-byte loads) and merges the ids that fall into the same word
// before calling `put` -- dense lists average several ids per word, so this cuts the global atomics behind `put` several-fold.
template <class Put>
IFX_FN void stream_list_words(const Ctx& c, const int32_t* list, int64_t n, Put put) {
    const int NT = c.nthreads(); int64_t done = 0;
    if (n >= 4096) {
        int64_t pre = (int64_t)((0 - (reinterpret_cast<uintptr_t>(list) >> 2)) & 3);     // ids in front of the first 16-byte boundary
        for (int64_t i = c.tid(); i < pre; i += NT) { int d = list[i]; put(d >> 5, 1u << (d & 31)); }
        struct alignas(16) Id4 { int32_t v[4]; };
        const Id4* p4 = reinterpret_cast<const Id4*>(list + pre); const int64_t n8 = (n - pre) >> 3;
        for (int64_t g0 = c.tid(); g0 < n8; g0 += 2LL * NT) {      // two runs (four loads) in flight per thread
            Id4 q[4]; const int64_t g1 = g0 + NT; const bool two = g1 < n8;
            q[0] = p4[2 * g0]; q[1] = p4[2 * g0 + 1]; if (two) { q[2] = p4[2 * g1]; q[3] = p4[2 * g1 + 1]; }
            for (int h = 0; h < (two ? 2 : 1); h++) {
                int word = q[2 * h].v[0] >> 5; unsigned mask = 0;
                for (int k = 0; k < 8; k++) { int d = q[2 * h + (k >> 2)].v[k & 3]; if ((d >> 5) != word) { put(word, mask); word = d >> 5; mask = 0; } mask |= 1u << (d & 31); }
                put(word, mask);
            }
        }
        done = pre + (n8 << 3);
    }
    const int64_t NT4 = 4LL * NT;
    for (int64_t i0 = done + c.tid(); i0 < n; i0 += NT4) {      // four independent loads in flight per thread
        int dd[4];
        for (int u = 0; u < 4; u++) { int64_t i = i0 + (int64_t)u * NT; dd[u] = i < n ? list[i] : -1; }
        for (int u = 0; u < 4; u++) if (dd[u] >= 0) put(dd[u] >> 5, 1u << (dd[u] & 31));
    }
}

// OR a sorted id list into the CTA's bitset; returns the number of newly set docs (block-wide).
IFX_FN int or_list_into_bits(const Ctx& c, const int32_t* list, int64_t n, S1Workspace& ws, S1SelShared& sh) {
    int fresh = 0;
    stream_list_words(c, list, n, [&](int word, unsigned mask) { unsigned old = atomic_or(&ws.bits[word], mask); fresh += popc(mask & ~old); sh.dirty[word >> 11] = 1; });
    c.sync();
    return block_sum(c, fresh, sh.scan);
}

// Warp-aggregated unordered append (all lanes of the warp must call it together).
IFX_FN void warp_append(const Ctx& c, bool pred, int32_t value, int32_t* arr, int* counter) {
    unsigned m = c.ballot(pred); if (m == 0) return;
    int leader = ffs32(m) - 1; int base = 0;
    if (c.lane() == leader) base = atomic_add(counter, popc(m));
    base = c.shfl(base, leader);
    if (pred) arr[base + popc(m & c.lanemask_lt())] = value;
}

// AND of the first `cnt` terms of sh.order (TieredCandidateSelector.IntersectTerms). The running intersection lives both as an
// unordered id array (ping-pong ws.buf_a / ws.buf_b) and as the membership bitset ws.bits2. Each further list either streams
// past the bitset (coalesced, when it is not much longer than the running set) or is probed per surviving id (binary search).
// Returns the size (-1: buffer overflow); `res` points at the surviving ids; ws.bits2 is left all-zero.
IFX_FN int64_t intersect_terms(const Ctx& c, const DevIndex& ix, S1Workspace& ws, S1SelShared& sh, int cnt, const int32_t*& res) {
    const int NT = c.nthreads();
    int by_len[MAX_TERMS];
    for (int i = 0; i < cnt; i++) by_len[i] = sh.order[i];
    for (int i = 1; i < cnt; i++) { int x = by_len[i]; int j = i - 1; while (j >= 0 && sh.terms[by_len[j]].len > sh.terms[x].len) { by_len[j + 1] = by_len[j]; j--; } by_len[j + 1] = x; }
    const TermS& t0 = sh.terms[by_len[0]];
    int64_t n = t0.len; if (n > ws.buf_cap) return -1;
    int32_t* cur = ws.buf_a; int32_t* nxt = ws.buf_b;
    const int bw = (int)(((int64_t)ix.n_docs + 31) >> 5);
    int li_start = 1; bool seeded = false;
    if (cnt > 1 && 4 * n >= bw && ws.buf_cap >= bw) {
        // Large running sets (>= 1/128 of the shard): keep the intersection as a bitset only. Lists with a membership bitmap are
        // ANDed word by word; the others (fuzzy unions, mid-size lists) are streamed against the bitset into a scratch bitmap
        // (buf_b) that then replaces it. No per-id probes or appends. As soon as the set has thinned out (< 1/512 of the shard) the
        // survivors are expanded into the id array and the remaining lists are probed per survivor below -- an AND over the 3-grams
        // of several words collapses after two or three lists, and streaming twenty more lists past a nearly empty bitset was the
        // most expensive part of the heaviest queries.
        unsigned* acc = ws.bits2; unsigned* tmp = reinterpret_cast<unsigned*>(nxt);
        if (t0.bm) { for (int w = c.tid(); w < bw; w += NT) acc[w] = t0.bm[w]; }
        else stream_list_words(c, t0.docs, t0.len, [&](int word, unsigned mask) { atomic_or(&acc[word], mask); });
        c.sync();
        auto expand = [&](bool clear) -> int64_t {
            int64_t total = 0;
            for (int w0 = 0; w0 < bw; w0 += 4 * NT) {
                unsigned v[4]; int mine = 0; const int wb = w0 + c.tid() * 4;
                for (int u = 0; u < 4; u++) { int w = wb + u; unsigned x = 0; if (w < bw) { x = acc[w]; if (clear) acc[w] = 0u; } v[u] = x; mine += popc(x); }
                int tot; int off = block_excl_scan(c, mine, sh.scan, tot);
                int64_t o = total + off;
                for (int u = 0; u < 4; u++) { unsigned x = v[u]; while (x) { int b = ffs32(x) - 1; x &= x - 1; cur[o++] = ((wb + u) << 5) | b; } }
                total += tot;
            }
            c.sync();
            return total;
        };
        for (int li = 1; li < cnt; li++) {
            const TermS& t = sh.terms[by_len[li]]; int mine = 0;
            if (t.bm) { for (int w = c.tid(); w < bw; w += NT) { const unsigned x = acc[w] & t.bm[w]; acc[w] = x; mine += popc(x); } }
            else {
                for (int w = c.tid(); w < bw; w += NT) tmp[w] = 0u;
                c.sync();
                stream_list_words(c, t.docs, t.len, [&](int word, unsigned mask) { unsigned hit = acc[word] & mask; if (hit) atomic_or(&tmp[word], hit); });
                c.sync();
                for (int w = c.tid(); w < bw; w += NT) { const unsigned x = tmp[w]; acc[w] = x; mine += popc(x); }
            }
            c.sync();
            const int64_t nbits = block_sum(c, mine, sh.scan);
            if (li + 1 < cnt && 16 * nbits < bw) { n = expand(false); li_start = li + 1; seeded = true; break; }      // bits2 keeps the membership: the invariant of the loop below
        }
        if (!seeded) { const int64_t total = expand(true); res = cur; return total; }
    }
    if (!seeded) {
        for (int64_t i = c.tid(); i < n; i += NT) { int d = t0.docs[i]; cur[i] = d; if (cnt > 1) atomic_or(&ws.bits2[d >> 5], 1u << (d & 31)); }
        c.sync();
    }
    for (int li = li_start; li < cnt && n > 0; li++) {
        const TermS& t = sh.terms[by_len[li]];
        if (c.tid() == 0) sh.bcast[6] = 0;
        c.sync();
        if (!t.bm && (int64_t)t.len <= 32 * n) {             // stream the list past the membership bitset (dense terms are probed through their bitmap instead)
            const int64_t rounds = ((int64_t)t.len + NT - 1) / NT;
            for (int64_t r = 0; r < rounds; r += 4) {         // four independent loads in flight per thread
                int64_t i0 = r * NT + c.tid(); int32_t d[4]; bool in[4];
                for (int u = 0; u < 4; u++) { int64_t i = i0 + (int64_t)u * NT; d[u] = (r + u < rounds && i < t.len) ? t.docs[i] : -1; }
                for (int u = 0; u < 4; u++) in[u] = d[u] >= 0 && ((ws.bits2[d[u] >> 5] >> (d[u] & 31)) & 1u);
                for (int u = 0; u < 4; u++) warp_append(c, in[u], d[u], nxt, &sh.bcast[6]);
            }
            c.sync();
            for (int64_t i = c.tid(); i < n; i += NT) { int d = cur[i]; atomic_and(&ws.bits2[d >> 5], ~(1u << (d & 31))); }   // drop the old set ...
            c.sync();
            const int64_t nn = sh.bcast[6];
            if (li + 1 < cnt) for (int64_t i = c.tid(); i < nn; i += NT) { int d = nxt[i]; atomic_or(&ws.bits2[d >> 5], 1u << (d & 31)); }   // ... keep the survivors
            n = nn;
        } else {                                              // probe the (much longer) list once per surviving id
            const int64_t rounds = (n + NT - 1) / NT;
            for (int64_t r = 0; r < rounds; r += 4) {        // four independent probes in flight per thread
                int dd[4]; bool found[4]; unsigned wv[4];
                for (int u = 0; u < 4; u++) { int64_t i = (r + u) * NT + c.tid(); dd[u] = (r + u < rounds && i < n) ? cur[i] : -1; }
                if (t.bm) { for (int u = 0; u < 4; u++) wv[u] = dd[u] >= 0 ? t.bm[dd[u] >> 5] : 0u; for (int u = 0; u < 4; u++) found[u] = dd[u] >= 0 && ((wv[u] >> (dd[u] & 31)) & 1u); }
                else for (int u = 0; u < 4; u++) { found[u] = false; if (dd[u] >= 0) { int d = dd[u]; int64_t lo = 0, hi = t.len; if (t.skip) { lo = t.skip[d >> 16]; hi = t.skip[(d >> 16) + 1]; } int64_t p = lower_bound_i32(t.docs, lo, hi, d); found[u] = p < hi && t.docs[p] == d; } }
                for (int u = 0; u < 4; u++) { if (dd[u] >= 0 && !found[u]) atomic_and(&ws.bits2[dd[u] >> 5], ~(1u << (dd[u] & 31))); if (r + u < rounds) warp_append(c, found[u], dd[u], nxt, &sh.bcast[6]); }
            }
            c.sync();
            n = sh.bcast[6];
            if (li + 1 == cnt) { for (int64_t i = c.tid(); i < n; i += NT) { int d = nxt[i]; atomic_and(&ws.bits2[d >> 5], ~(1u << (d & 31))); } }
        }
        c.sync();
        int32_t* tmp = cur; cur = nxt; nxt = tmp;
    }
    if (cnt > 1 && n == 0) { /* bitset already empty: every id was cleared when it dropped out */ }
    res = cur;
    c.sync();
    return n;
}

// Expand the dirty containers of the bitset into ws.cand (ascending) and clear them. Returns the count.
IFX_FN int64_t compact_bits(const Ctx& c, const DevIndex& ix, S1Workspace& ws, S1SelShared& sh, int32_t* out, int64_t out_cap, bool& overflow) {
    int ncont = (ix.n_docs + 65535) >> 16; int64_t total = 0; int64_t nwords = ((int64_t)ix.n_docs + 31) >> 5;
    overflow = false;
    for (int k = 0; k < ncont; k++) {
        if (!sh.dirty[k]) continue;                    // uniform across the CTA (shared flag, synced by callers)
        int64_t w0 = (int64_t)k * 2048, w1 = w0 + 2048; if (w1 > nwords) w1 = nwords;
        int per = (int)((w1 - w0 + c.nthreads() - 1) / c.nthreads());
        int64_t my0 = w0 + (int64_t)c.tid() * per, my1 = my0 + per; if (my1 > w1) my1 = w1;
        int cnt = 0; for (int64_t w = my0; w < my1; w++) cnt += popc(ws.bits[w]);
        int tot; int off = block_excl_scan(c, cnt, sh.scan, tot);
        if (total + tot > out_cap) { overflow = true; }
        else { int64_t o = total + off;
            for (int64_t w = my0; w < my1; w++) { unsigned v = ws.bits[w]; while (v) { int b = ffs32(v) - 1; out[o++] = (int32_t)((w << 5) | b); v &= v - 1; } } }
        for (int64_t w = my0; w < my1; w++) ws.bits[w] = 0;
        total += tot;
        c.sync();
        if (c.tid() == 0) sh.dirty[k] = 0;
    }
    c.sync();
    return total;
}

// .NET ArraySortHelper<T>.IntrospectiveSort with comparison (b.Idf.CompareTo(a.Idf)) over term indices -- unstable,
// reproduced exactly because idf ties decide which lists the selector unions (TieredCandidateSelector.cs:128,253).
struct IdfSorter {
    const TermS* t;
    IFX_FN int cmp(int a, int b) const { float x = t[b].idf, y = t[a].idf; return x < y ? -1 : (x > y ? 1 : 0); }
    IFX_FN void swap_if_greater(int* k, int i, int j) const { if (cmp(k[i], k[j]) > 0) { int x = k[i]; k[i] = k[j]; k[j] = x; } }
    IFX_FN void insertion(int* k, int n) const { for (int i = 0; i < n - 1; i++) { int t2 = k[i + 1]; int j = i; while (j >= 0 && cmp(t2, k[j]) < 0) { k[j + 1] = k[j]; j--; } k[j + 1] = t2; } }
    IFX_FN void down_heap(int* k, int i, int n) const { int d = k[i - 1]; while (i <= n / 2) { int ch = 2 * i; if (ch < n && cmp(k[ch - 1], k[ch]) < 0) ch++; if (!(cmp(d, k[ch - 1]) < 0)) break; k[i - 1] = k[ch - 1]; i = ch; } k[i - 1] = d; }
    IFX_FN void heap_sort(int* k, int n) const { for (int i = n >> 1; i >= 1; i--) down_heap(k, i, n); for (int i = n; i > 1; i--) { int x = k[0]; k[0] = k[i - 1]; k[i - 1] = x; down_heap(k, 1, i - 1); } }
    IFX_FN int partition(int* k, int n) const {
        int hi = n - 1, mid = hi >> 1;
        swap_if_greater(k, 0, mid); swap_if_greater(k, 0, hi); swap_if_greater(k, mid, hi);
        int pivot = k[mid]; { int x = k[mid]; k[mid] = k[hi - 1]; k[hi - 1] = x; }
        int left = 0, right = hi - 1;
        while (left < right) {
            while (cmp(k[++left], pivot) < 0) {}
            while (cmp(pivot, k[--right]) < 0) {}
            if (left >= right) break;
            int x = k[left]; k[left] = k[right]; k[right] = x;
        }
        if (left != hi - 1) { int x = k[left]; k[left] = k[hi - 1]; k[hi - 1] = x; }
        return left;
    }
    IFX_FN void sort(int* keys, int n) const {
        if (n < 2) return;
        int lg = 0; for (unsigned v = (unsigned)n; v >>= 1;) lg++;
        // explicit stack instead of recursion: (start, length, depth)
        int st_s[64], st_n[64], st_d[64]; int sp = 0; st_s[0] = 0; st_n[0] = n; st_d[0] = 2 * (lg + 1); sp = 1;
        while (sp > 0) {
            sp--; int* k = keys + st_s[sp]; int len = st_n[sp], depth = st_d[sp]; int s0 = st_s[sp];
            while (len > 1) {
                if (len <= 16) { if (len == 2) swap_if_greater(k, 0, 1); else if (len == 3) { swap_if_greater(k, 0, 1); swap_if_greater(k, 0, 2); swap_if_greater(k, 1, 2); } else insertion(k, len); break; }
                if (depth == 0) { heap_sort(k, len); break; }
                depth--;
                int p = partition(k, len);
                // reference recurses into the right part first, then loops on the left part; the two parts are disjoint so order is irrelevant
                st_s[sp] = s0 + p + 1; st_n[sp] = len - (p + 1); st_d[sp] = depth; sp++;
                len = p;
            }
        }
    }
};

// .NET PriorityQueue<int,float> (4-ary min-heap) on shared arrays -- Bm25Scorer.UpdateTopK (Bm25Scorer.cs:654-670)
IFX_FN float kv_score(unsigned long long kv) {
#ifdef IFX_EMU
    unsigned u = (unsigned)kv; float f; memcpy(&f, &u, 4); return f;
#else
    return __uint_as_float((unsigned)kv);
#endif
}
IFX_FN unsigned long long kv_pack(int doc, float pr) {
#ifdef IFX_EMU
    unsigned u; memcpy(&u, &pr, 4); return ((unsigned long long)(unsigned)doc << 32) | u;
#else
    return ((unsigned long long)(unsigned)doc << 32) | __float_as_uint(pr);
#endif
}
#define IFX_HP(i) heap_pr[(i) + 3]
#define IFX_HD(i) heap_doc[(i) + 3]
template <class H> IFX_FN void heap_move_up(H& sh, int doc, float pr, int idx) {
    while (idx > 0) { int parent = (idx - 1) >> 2; float pp = sh.IFX_HP(parent); if (pr < pp) { sh.IFX_HP(idx) = pp; sh.IFX_HD(idx) = sh.IFX_HD(parent); idx = parent; } else break; }
    sh.IFX_HP(idx) = pr; sh.IFX_HD(idx) = doc;
}
// PriorityQueue.DequeueEnqueue on a full heap (the root is replaced and sifted down); returns the new root priority so the caller
// can keep the threshold in a register. PriorityQueue.MoveDown picks the first strictly-smallest of the (up to) four children; here as
// a two-level tournament with the same winner (ties keep the lower index at both levels). Only the priorities are on the
// dependent chain; the document id of a moved node follows with one load/store off it.
template <class H> IFX_FN float heap_replace_root(H& sh, int doc, float pr, int sz) {
    int idx = 0, i; float root = pr;
    while ((i = 4 * idx + 1) < sz) {
#ifdef IFX_EMU
        const float p0 = sh.IFX_HP(i), p1 = sh.IFX_HP(i + 1), p2 = sh.IFX_HP(i + 2), p3 = sh.IFX_HP(i + 3);
#else
        const float4 v = *reinterpret_cast<const float4*>(&sh.heap_pr[i + 3]); const float p0 = v.x, p1 = v.y, p2 = v.z, p3 = v.w;
#endif
        const bool b01 = p1 < p0, b23 = p3 < p2; const float pa = b01 ? p1 : p0, pb = b23 ? p3 : p2;
        const bool bb = pb < pa; const float mp = bb ? pb : pa; const int mi = i + (bb ? (b23 ? 3 : 2) : (b01 ? 1 : 0));
        if (!(mp < pr)) break;
        sh.IFX_HP(idx) = mp; sh.IFX_HD(idx) = sh.IFX_HD(mi); if (idx == 0) root = mp;
        idx = mi;
    }
    sh.IFX_HP(idx) = pr; sh.IFX_HD(idx) = doc;
    return root;
}

// Bm25Scorer.cs:395-433 (Vector256 lanes) and :643-652 (scalar remainder); must not be contracted into FMAs.
// The document-length part of both forms depends only on the candidate, so it is evaluated once per chunk and slot:
//   vector form  norm = K1 * ((1 - B) + (B / avgdl) * dl)        (the scalar form, needed for < 8 matches per term and chunk, is recomputed)
IFX_FN float bm25_norm_vector(float dl, float avgdl) { const float K1 = 1.2f, B = 0.75f; float bdiv = B / avgdl; return K1 * ((1.f - B) + bdiv * dl); }
IFX_FN float bm25_from_norm_vector(float tf, float norm, float idf) { const float K1 = 1.2f, Delta = 1.0f; float denom = tf + norm; float core = (tf * (K1 + 1.0f)) / denom; return idf * (core + Delta); }
IFX_FN float bm25_scalar(float tf, float dl, float avgdl, float idf) {
    const float K1 = 1.2f, B = 0.75f, Delta = 1.0f;
    if (dl <= 0.f) dl = 1.f;
    float norm = K1 * (1.f - B + B * (dl / avgdl)); float denom = tf + norm;
    if (denom <= 0.f) return 0.f;
    float core = (tf * (K1 + 1.f)) / denom; return idf * (core + Delta);
}

struct Stage1Out { int64_t* key; int32_t* doc; float* score; int32_t* n; long long* dbg; };   // dbg: [n_cand, n_terms, selection ns, path] or null   // row pointers for this query (cap = depth)

// ---------------------------------------------------------------------------------------------------------------
// LD1 expansion of one unknown word: first 1024 trie-order matches (Myers bit-vector, search variant), union of
// their posting lists -> ascending unique doc list appended to the fuzzy pool.
IFX_FN void expand_fuzzy(const Ctx& c, const DevIndex& ix, QueryPlan& p, int fslot, S1Workspace& ws, S1Shared& sh,
                         int32_t* pool, unsigned long long pool_cap, BatchCounters* bc, const uint8_t* sorted_len, int32_t* matches /* [LD1_CAP] global or shared */) {
    const FuzzyReq fr = p.fuzzy[fslot];
    const uint16_t* q = p.ttext + fr.off; const int m = fr.len;
    const uint64_t maskM = 1ULL << (m - 1);
    int64_t T = ix.terms.n; int total = 0;
    // a term within (search-variant) edit distance 1 of the word lacks at most one of the word's distinct characters
    const unsigned long long qsig = char_sig(q, m);
    for (int ch = c.tid(); ch < 128; ch += c.nthreads()) { unsigned long long pm = 0; for (int j = 0; j < m; j++) if (q[j] == ch) pm |= 1ULL << j; sh.peq[ch] = pm; }
    c.sync();
    // Myers bit-vector (search variant, FstIndex.cs:316-335) along one dictionary term (ordinal `ord`, length L)
    auto myers_hit = [&](int ord, int L) -> bool {
        const uint16_t* s = ix.terms.chars + ix.terms.off[ord];
        uint64_t vp = ~0ULL, vn = 0ULL; int score = m;
        for (int k = 0; k < L; k++) {
            uint16_t ch = s[k]; uint64_t pm;
            if (ch < 128) pm = sh.peq[ch]; else { pm = 0; for (int j = 0; j < m; j++) if (q[j] == ch) pm |= 1ULL << j; }
            uint64_t x = pm | vn; uint64_t d0 = ((vp + (x & vp)) ^ vp) | x; uint64_t hn = vp & d0; uint64_t hp = vn | ~(vp | d0);
            uint64_t nvp = (hn << 1) | ~(d0 | (hp << 1)); uint64_t nvn = d0 & (hp << 1);
            if (hp & maskM) score++; if (hn & maskM) score--;
            vp = nvp; vn = nvn;
        }
        return score <= 1;
    };
    {   // Fast path: only dictionary terms of length m-1..m+1 can match, and the dictionary is also stored grouped by length
        // (ix.len_ptr / len_sig / len_ord), so the scan is a coalesced stream over those three groups. Matches are appended in
        // arbitrary order: the union below is order-free as long as all of them fit (<= LD1_CAP, the usual case).
        if (c.tid() == 0) sh.bcast[6] = 0;
        c.sync();
        const int l0 = m - 1 < 0 ? 0 : m - 1, l1 = m + 1 > 254 ? 254 : m + 1;
        const int64_t gb = ix.len_ptr[l0], ge = l1 >= l0 ? ix.len_ptr[l1 + 1] : gb; const int64_t g1 = ix.len_ptr[l0 + 1], g2 = l0 + 2 <= 255 ? ix.len_ptr[l0 + 2] : ge;
        const int64_t NT4 = 4LL * c.nthreads();
        for (int64_t base0 = gb; base0 < ge; base0 += NT4) {       // uniform trip count (warp votes inside); four signature loads in flight per thread
            const int64_t i0 = base0 + c.tid(); unsigned long long sg[4];
            for (int u = 0; u < 4; u++) { int64_t i = i0 + (int64_t)u * c.nthreads(); sg[u] = i < ge ? ix.len_sig[i] : ~0ULL; }
            for (int u = 0; u < 4; u++) {
                int64_t i = i0 + (int64_t)u * c.nthreads(); bool hit = false; int ord = 0;
                if (i < ge && popc64(qsig & ~sg[u]) <= 1) { ord = ix.len_ord[i]; int L = l0 + (i >= g1 ? 1 : 0) + (i >= g2 ? 1 : 0); hit = myers_hit(ord, L); }
                unsigned bm = c.ballot(hit);
                if (bm) { int leader = ffs32(bm) - 1; int base = 0; if (c.lane() == leader) base = atomic_add(&sh.bcast[6], popc(bm)); base = c.shfl(base, leader);
                          int at = base + popc(bm & c.lanemask_lt()); if (hit && at < LD1_CAP) matches[at] = ord; }
            }
        }
        c.sync();
        total = sh.bcast[6];
        c.sync();
        if (total > LD1_CAP) {
            // more matches than VectorModel.cs:662 keeps: the reference takes the first LD1_CAP in trie DFS order, so redo the scan
            // over the lexicographically sorted dictionary with an ordered compaction and stop there
            total = 0;
            for (int64_t base = 0; base < T && total < LD1_CAP; base += c.nthreads()) {
                int64_t i = base + c.tid(); bool hit = false;
                if (i < T) { int L = sorted_len[i]; hit = L >= m - 1 && L <= m + 1 && L < 255 && popc64(qsig & ~ix.term_sig[i]) <= 1 && myers_hit(ix.term_sorted[i], L); }
                int t2; int o2 = block_excl_scan(c, hit ? 1 : 0, sh.scan, t2);
                if (hit && total + o2 < LD1_CAP) matches[total + o2] = ix.term_sorted[i];
                total += t2;
            }
        }
    }
    c.sync();
    const int nm = total < LD1_CAP ? total : LD1_CAP;
    // Union of the matches' posting lists into the CTA's bitset: short lists one warp each (no block barrier per list), long
    // lists block-wide afterwards.
    const int BIG = 4096, BIGQ = 128; int fresh = 0;
    if (c.tid() == 0) sh.bcast[5] = 0;
    c.sync();
    for (int k = c.warp(); k < nm; k += c.nwarps()) {
        int ord = matches[k]; if (ix.df[ord] <= 0) continue;
        int64_t r0 = ix.row_ptr[ord], r1 = ix.row_ptr[ord + 1];
        if (r1 - r0 >= BIG) { int slot = BIGQ; if (c.lane() == 0) slot = atomic_add(&sh.bcast[5], 1); slot = c.shfl(slot, 0); if (slot < BIGQ) { if (c.lane() == 0) sh.bprefix[slot] = ord; continue; } }
        for (int64_t i = r0 + c.lane(); i < r1; i += Ctx::WS) {
            int d = ix.post_doc[i]; unsigned bit = 1u << (d & 31);
            unsigned old = atomic_or(&ws.bits[d >> 5], bit);
            if (!(old & bit)) fresh++;
            sh.dirty[d >> 16] = 1;
        }
    }
    c.sync();
    int df = block_sum(c, fresh, sh.scan);
    const int nbig = sh.bcast[5] < BIGQ ? sh.bcast[5] : BIGQ;
    for (int k = 0; k < nbig; k++) { int ord = sh.bprefix[k]; int64_t r0 = ix.row_ptr[ord], r1 = ix.row_ptr[ord + 1]; df += or_list_into_bits(c, ix.post_doc + r0, r1 - r0, ws, sh); }
    c.sync();
    QTerm& t = p.terms[fr.term_slot];
    if (df == 0) { if (c.tid() == 0) { t.df = 0; t.list_len = 0; } c.sync(); return; }
    if (c.tid() == 0) { unsigned long long b = atomic_add64(&bc->fuzzy_pool_used, (unsigned long long)df); sh.bcast64[0] = (long long)b; }
    c.sync();
    unsigned long long b = (unsigned long long)sh.bcast64[0]; bool ovf = false;
    int64_t cap = b + (unsigned long long)df <= pool_cap ? df : 0;
    int64_t n = compact_bits(c, ix, ws, sh, pool + b, cap, ovf);
    if (c.tid() == 0) {
        if (ovf || n != df) { p.status |= 4; atomic_add(&bc->overflow, 1); t.df = 0; t.list_len = 0; }
        else { float avgdl = ix.avgdl > 0.f ? ix.avgdl : 1.f; t.df = df; t.list_len = df; t.list_off = (int64_t)b; t.idf = compute_idf(ix, df); t.max_score = max_term_score(t.idf, avgdl); }
    }
    c.sync();
}

// Prefix precedence (TieredCandidateSelector.TrySelectPrefixCandidates): the candidates are the doc set of the query's first 1-3
// characters when that set is small enough. Returns its range in ix.prefix.doc_id.
IFX_FN bool prefix_shortcut(const DevIndex& ix, const QueryPlan& p, int K, int64_t& r0, int64_t& pop) {
    int maxl = p.tlen < 3 ? p.tlen : 3;
    for (int len = maxl; len >= 1; len--) {
        int k = dict_lookup(ix.prefix.keys, p.ttext, len); if (k < 0) continue;
        r0 = ix.prefix.row_ptr[k]; const int64_t local = ix.prefix.row_ptr[k + 1] - r0; pop = ix.prefix_gcard ? (int64_t)ix.prefix_gcard[k] : local;      // the rules look at the cardinality over the whole corpus
        if (pop == 0) continue;
        if (pop > (int64_t)K * 20) continue;
        if (pop <= (int64_t)K * 10) { int lim = K * 2 < 100 ? K * 2 : 100; const bool take = pop >= lim; pop = local; return take; }      // candidates: this shard's part of the set
    }
    return false;
}

// ---------------------------------------------------------------------------------------------------------------
// Candidate selection of one query (TieredCandidateSelector.SelectCandidates). Leaves the candidate set as bits in ws.bits (dirty
// containers flagged in sh.dirty), the scored terms in sh.terms / sh.n_terms; `path`: 0 nothing to score, 1 prefix shortcut, 2 disjunctive,
// 3 AND tiers, -1 workspace overflow.
// Doc-id-range shards (`smode`): the tier rules compare CORPUS-level cardinalities, so a shard first runs the selection in count mode
// (smode 1: local cardinality at every decision point into cnt[], following every branch that some shard might need), the hosts sum the
// counts over the shards, and the real pass (smode 2) takes its decisions from the global values in cnt[]. smode 0: unsharded.
constexpr int SEL_CNT = 40;          // cnt[0..3]: AND path (tier 0, + tier 1, + first / second high-idf list); cnt[8 + i]: disjunctive path after list i (i < 32)
                                     // cnt[4]: count pass only -- 1 when every decision was forced by this shard's own count (local >= limit implies corpus >= limit): the
                                     // candidate set is already final and the shard goes straight on to the lookups; (kept per shard in a separate flag array, not summed)
IFX_FN int stage1_select(const Ctx& c, const DevIndex& ix, const QueryPlan& p, const int32_t* pool, S1Workspace& ws, S1SelShared& sh, Stage1Out out, int smode = 0, int32_t* cnt = nullptr) {
    const int K = p.depth; const int NT = c.nthreads();
    if (c.tid() == 0) {
        int n = 0;
        for (int i = 0; i < p.n_terms; i++) {
            const QTerm& q = p.terms[i];
            if (q.df <= 0 || q.df > ix.stop_term_limit) continue;      // VectorModel.cs:521
            TermS& t = sh.terms[n]; t.len = q.list_len; t.df = q.df; t.idf = q.idf; t.max_score = q.max_score; t.cursor = 0; t.term_id = q.term_id;
            if (q.term_id >= 0) { t.docs = ix.post_doc + q.list_off; t.tf = ix.post_tf + q.list_off; int sk = ix.skip_id[q.term_id]; t.skip = sk >= 0 ? ix.skip_ptr + (size_t)sk * (ix.n_cont + 1) : nullptr;
                int bi = ix.bm_id[q.term_id]; t.bm = bi >= 0 ? ix.bm_bits + (size_t)bi * ix.bm_words : nullptr; t.bmr = bi >= 0 ? ix.bm_rank + (size_t)bi * ix.bm_words : nullptr; }
            else { t.docs = pool + q.list_off; t.tf = nullptr; t.skip = nullptr; t.bm = nullptr; t.bmr = nullptr; }
            n++;
        }
        float suf = 0.f; for (int i = n - 1; i >= 0; i--) { sh.terms[i].suffix_after = suf; suf = suf + sh.terms[i].max_score; }   // ComputeSuffixSums
        for (int i = 0; i < QH_SIZE; i++) sh.qh_key[i] = -1;
        for (int i = 0; i < n; i++) { const TermS& t = sh.terms[i]; if (t.term_id < 0 || t.idf <= 0.f) continue;      // (ids are unique within a query)
            unsigned h = qh_hash(t.term_id); while (sh.qh_key[h] >= 0) h = (h + 1) & (QH_SIZE - 1); sh.qh_key[h] = t.term_id; sh.qh_slot[h] = (uint8_t)i; }
        sh.n_terms = n; sh.streamed_mask[0] = sh.streamed_mask[1] = 0;
        out.n[0] = 0;
    }
    c.sync();
    const int T = sh.n_terms;
    if (T == 0 || ix.n_live == 0 || p.status != 0) return 0;

    // ---- candidate selection (TieredCandidateSelector.SelectCandidates)
#if !defined(IFX_EMU) && defined(IFX_S1_TIMERS)
    long long smark = 0; if (c.tid() == 0) { asm volatile("mov.u64 %0, %%clock64;" : "=l"(smark) :: "memory"); if (out.dbg) for (int k = 20; k < 24; k++) out.dbg[k] = 0; }
#define IFX_STICK(k) do { c.sync(); if (c.tid() == 0 && out.dbg) { long long now_; asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_) : "r"(sh.bcast[0]) : "memory"); out.dbg[20 + (k)] += now_ - smark; smark = now_; } } while (0)
#else
#define IFX_STICK(k) do { } while (0)
#endif
    int path = 0; bool certain = false;
    if (c.tid() == 0) { sh.bcast64[0] = -1; sh.bcast64[1] = 0; int64_t r0, pop; if (prefix_shortcut(ix, p, K, r0, pop)) { sh.bcast64[0] = r0; sh.bcast64[1] = pop; } }
    c.sync();
    if (sh.bcast64[0] >= 0) { path = 1; certain = true; or_list_into_bits(c, ix.prefix.doc_id + sh.bcast64[0], sh.bcast64[1], ws, sh); }      // (the prefix rules read replicated corpus-level cardinalities)
    else {
        if (c.tid() == 0) {
            bool typo = false; float max_idf = 0.f;
            for (int i = 0; i < T; i++) { if (sh.terms[i].df < 10) typo = true; if (sh.terms[i].idf > max_idf) max_idf = sh.terms[i].idf; sh.order[i] = i; }
            IdfSorter srt{sh.terms}; srt.sort(sh.order, T);
            sh.bcast[0] = (typo || T == 1) ? 1 : 0; ((float*)sh.bcast)[1] = max_idf;
        }
        c.sync();
        const bool disjunctive = sh.bcast[0] != 0; const float max_idf = ((float*)sh.bcast)[1];
        int64_t g = 0;
        IFX_STICK(0);   // prefix shortcut + idf sort
        if (disjunctive) {   // SelectCandidatesDisjunctive
            bool selective = false; int li = 0; int64_t df_max = 0; if (smode == 1 && T == 1) certain = true;      // a single list: nothing to decide
            for (int oi = 0; oi < T; oi++) {
                const TermS& t = sh.terms[sh.order[oi]];
                bool lowq = t.idf < (max_idf * 0.2f);
                if (T > 1 && lowq && selective) continue;
                g += or_list_into_bits(c, t.docs, t.len, ws, sh);
                if (c.tid() == 0) sh.streamed_mask[sh.order[oi] >> 6] |= 1ULL << (sh.order[oi] & 63);
                int64_t gg = g;                                                   // the union's size over the whole corpus decides
                if (smode == 1 && li < 32) { if (c.tid() == 0) cnt[8 + li] = (int32_t)g; if (t.df > df_max) df_max = t.df; gg = df_max;      // count pass: go on until the union certainly holds 100 K documents (it contains its largest list)
                    if (g >= (int64_t)K * 100 && li == 0) { certain = true; gg = g; } }                                                      // ... or, at the very first list, stop for good: this shard alone has them
                else if (smode == 2 && li < 32) gg = cnt[8 + li];
                li++;
                if (!lowq && gg > 0) selective = true;
                if (gg >= (int64_t)K * 100) break;
            }
        } else {
            if (c.tid() == 0) for (int i = 0; i < T; i++) sh.streamed_mask[i >> 6] |= 1ULL << (i & 63);   // every list of the AND tier
            const int32_t* r0 = nullptr; int64_t n0 = intersect_terms(c, ix, ws, sh, T, r0);
            if (n0 < 0) { if (c.tid() == 0) out.n[0] = -1; return -1; }
            g += or_list_into_bits(c, r0, n0, ws, sh);
            IFX_STICK(1);   // AND tier 0
            // count pass: a shard that alone reaches a limit knows the corpus does; below it every later stage is counted (some shard may need it)
            int64_t G = smode == 2 ? (int64_t)cnt[0] : g; if (smode == 1 && c.tid() == 0) { cnt[0] = (int32_t)g; cnt[1] = cnt[2] = cnt[3] = (int32_t)g; }
            if (smode == 1 && g >= (int64_t)K * 2) certain = true;          // tier 0 alone is enough on this shard, hence in the corpus
            if (G < (int64_t)K * 2) {
                if (T >= 3 && G < (int64_t)K * 3) { const int32_t* r1 = nullptr; int64_t n1 = intersect_terms(c, ix, ws, sh, T - 1, r1); if (n1 > 0) g += or_list_into_bits(c, r1, n1, ws, sh); }
                IFX_STICK(2);   // AND tier 1
                G = smode == 2 ? (int64_t)cnt[1] : g; if (smode == 1 && c.tid() == 0) { cnt[1] = (int32_t)g; cnt[2] = cnt[3] = (int32_t)g; }
                if (G < (int64_t)K * 5) {
                    int sel[2]; int ns = 0; float cutoff = max_idf * 0.3f; int capn = T < 2 ? T : 2;
                    for (int oi = 0; oi < T && ns < capn; oi++) { const TermS& t = sh.terms[sh.order[oi]]; if (t.idf <= 0.f) continue; if (t.idf < cutoff) continue; sel[ns++] = sh.order[oi]; }
                    for (int si = 0; si < ns; si++) { const TermS& t = sh.terms[sel[si]]; g += or_list_into_bits(c, t.docs, t.len, ws, sh);
                        G = smode == 2 ? (int64_t)cnt[2 + si] : g; if (smode == 1 && c.tid() == 0) { cnt[2 + si] = (int32_t)g; if (si == 0) cnt[3] = (int32_t)g; }
                        if (G >= (int64_t)K * 10) break; }
                }
            }
        }
        IFX_STICK(1);   // list unions (disjunctive: everything; AND path: the top-idf lists after the tiers)
        path = disjunctive ? 2 : 3;
    }
    if (smode == 1 && c.tid() == 0) cnt[4] = certain ? 1 : 0;
    if (c.tid() == 0 && out.dbg) { out.dbg[1] = T; out.dbg[3] = path;
#ifndef IFX_EMU
        unsigned long long tn; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tn)); out.dbg[2] = (long long)tn;
#endif
    }
    return path;
}

// Candidate bitset back to all-zero (dirty containers only).
IFX_FN void stage1_clear_bits(const Ctx& c, const DevIndex& ix, S1Workspace& ws, S1SelShared& sh) {
    const int NT = c.nthreads(); const int64_t nwords = ((int64_t)ix.n_docs + 31) >> 5; const int ncont = (ix.n_docs + 65535) >> 16;
    c.sync();
    for (int64_t w = c.tid(); w < nwords; w += NT) if (sh.dirty[w >> 11]) ws.bits[w] = 0u;
    c.sync();
    for (int k = c.tid(); k < ncont; k += NT) sh.dirty[k] = 0;
    c.sync();
}

}  // namespace ifx
