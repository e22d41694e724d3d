// infidex_b200 -- Stage 1 after candidate selection: tf lookups for ALL candidates of a query in one throughput-oriented pass
// (stage1_lookup, same CTA as the selection), then the order-dependent part -- BM25+ with MaxScore over the reference's chunks and the
// exact replay of its pruning heap (Bm25Scorer.cs:195-445,654-670) -- as a lean chain over pre-staged data:
//   score_warp  one WARP per query (queries whose chunks hold <= W_CAP candidates: the common case on large corpora, where a query's
//               candidates spread thinly over many 65 536-doc containers) -- thousands of independent chains per GPU, no block barrier
//   score_cta   one CTA per query (dense chunks, up to 4096 candidates): the tiled block-wide scorer
//   s1_finish   TopKHeap.GetTopK + ConsolidateSegments order (score desc, key asc) of the surviving heap
// What is staged per query in the batch's pool (S1Rec): candidate ids (ascending; bit 31 = deleted document), their document lengths,
// the chunk table (container runs cut into sub-chunks of 4096, Bm25Scorer.cs:209-270), per-term constants, and the tf matrix stored
// chunk-major ([term][slot] per chunk, rows padded to 16 bytes) so that a chunk is ONE contiguous, 16-byte aligned block.
#pragma once
#include "ifx_stage1.h"

namespace ifx {

struct S1Chunk { int32_t start, cnt; int64_t tf_off; };                       // tf_off: bytes from the query's tf base
struct S1TermP { float idf, max_score, suffix_after; int32_t pad; };
struct S1Rec {
    int64_t off_cand, off_dl, off_tf, off_chunk, off_terms;                    // byte offsets into the batch pool
    int32_t n_cand, n_chunks, n_terms, max_cnt;
    int32_t state;                                                            // 0 nothing to score, 1 light / 4 mid (score_warp), 3 heavy (score_cta), 2 deferred (pool full), -1 overflow
    int32_t K, path, pad;
};
struct S1Queues { int32_t* light; int32_t* mid; int32_t* heavy; };            // query ids appended by stage1_lookup (counters in BatchCounters)
struct alignas(16) S1Cont { int32_t cstart, cnt, cpad, cfirst; };                // per container: candidates before it, its candidates, padded tf slots before it, chunks before it

// Shared memory of the selection / tf-lookup kernel: the selection's state plus the on-chip slice of the candidate bitset that the
// streamed tf lookups probe, one 65 536-doc container at a time. (A struct of its own: S1Shared, the scorer's and the LD1
// expansion's at two CTAs per SM, extends S1SelShared and has no room for the slice.)
constexpr int CONT_WORDS = 65536 / 32;
struct S1LookShared : S1SelShared {
    unsigned cbits[CONT_WORDS];                // the container's bitset words
    uint16_t crank[CONT_WORDS];                // the container's candidates before each word
    const int32_t* sdoc[MAX_TERMS]; const uint8_t* stf[MAX_TERMS];   // streamed list j: its postings (and tfs) in the container, from the first one on
    int slen[MAX_TERMS]; int spre[MAX_TERMS + 1];                      // ... smis + their count, and where they start in the container's flattened range
    uint8_t smis[MAX_TERMS], slist[MAX_TERMS], srow[MAX_TERMS];        // ... 16-byte misalignment of the first (in postings), its slot in `terms`, its row of the tf matrix
};

IFX_FN int pad16(int x) { return (x + 15) & ~15; }
constexpr int DEL_BIT = (int)0x80000000;

// warp-scorer limits: a query is scored by one warp when its largest chunk holds <= W_CAP_MID candidates, it has <= W_TERMS scored terms
// and its depth fits the per-warp heap; "light" (<= W_CAP candidates per chunk: 8 slots per lane) and "mid" (16 slots per lane)
constexpr int W_CAP = 256, W_CAP_MID = 512;
constexpr int W_TF = 6144;           // bytes of the per-warp tf staging buffer (one tile of term rows of the current chunk)
constexpr int W_TERMS = 64;
constexpr int W_K = 512;             // heap capacity kept in shared memory per warp

// ---------------------------------------------------------------------------------------------------------------
// stage1_lookup: called right after stage1_select by the same CTA. Candidates are the bits of ws.bits.
//   1. count + expand the bitset into the pool (ascending ids), candidates before every container
//   2. document lengths, deleted flags, chunk table
//   3. tf of every (term, candidate): either every posting list streamed once against the candidate bitset (coalesced; the byte
//      volume SURVEY 8d calls algorithmic), or -- few candidates relative to the lists -- one forward-index read per candidate.
//      The lists are streamed container by container: the container's 8 KB of bitset and its per-word candidate ranks sit in shared
//      memory, so a posting's probe never leaves the SM
//   4. bitset cleared again
IFX_FN void stage1_lookup(const Ctx& c, const DevIndex& ix, const QueryPlan& p, int path, int q, S1Workspace& ws, S1LookShared& sh, S1Rec* recs,
                          unsigned char* spool, unsigned long long spool_cap, S1Queues queues, BatchCounters* bc, Stage1Out out, int fwd_avg_bytes, int force_mode) {
    S1Rec& rec = recs[q]; const int NT = c.nthreads(), NW = c.nwarps(); constexpr int WS = Ctx::WS;
#if !defined(IFX_EMU) && defined(IFX_S1_TIMERS)
    long long lmark = 0; if (c.tid() == 0) { asm volatile("mov.u64 %0, %%clock64;" : "=l"(lmark) :: "memory"); if (out.dbg) for (int k = 11; k < 18; k++) out.dbg[k] = 0; }
#define IFX_LTICK(k) do { c.sync(); if (c.tid() == 0 && out.dbg) { long long now_; asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_) :: "memory"); out.dbg[11 + (k)] += now_ - lmark; lmark = now_; } } while (0)
#else
#define IFX_LTICK(k) do { } while (0)
#endif
    if (path <= 0) { if (c.tid() == 0) { rec.state = path < 0 ? -1 : 0; rec.n_cand = 0; rec.K = p.depth; rec.path = path; } c.sync(); return; }
    const int T = sh.n_terms; const int64_t nwords = ((int64_t)ix.n_docs + 31) >> 5; const int ncont = (ix.n_docs + 65535) >> 16;
    // ---- 1a. count (each warp owns a contiguous span of bitset words; non-dirty containers are skipped)
    const int64_t span = (((nwords + NW - 1) / NW) + 31) / 32 * 32; const int64_t w0 = (int64_t)c.warp() * span, w1 = w0 + span < nwords ? w0 + span : nwords;
    int mycnt = 0;
    for (int64_t g0 = w0; g0 < w1; g0 += 4 * WS) {      // four groups (independent loads) per trip
        unsigned v[4];
        for (int u = 0; u < 4; u++) { const int64_t g = g0 + u * WS, w = g + c.lane(); v[u] = (g < w1 && sh.dirty[g >> 11] && w < w1) ? ws.bits[w] : 0u; }
        for (int u = 0; u < 4; u++) mycnt += popc(v[u]);
    }
    int n_cand; int ex0 = block_excl_scan(c, mycnt, sh.scan, n_cand); const int wbase = c.shfl(ex0, 0);
    auto clear_bits = [&]() {
        for (int64_t w = c.tid(); w < nwords; w += NT) if (sh.dirty[w >> 11]) ws.bits[w] = 0u;
        c.sync();
        for (int k = c.tid(); k < ncont; k += NT) sh.dirty[k] = 0;
        c.sync();
    };
    if (n_cand == 0) { clear_bits(); if (c.tid() == 0) { rec.state = 0; rec.n_cand = 0; rec.K = p.depth; rec.path = path; if (out.dbg) out.dbg[0] = 0; } c.sync(); return; }
    auto pool_alloc = [&](unsigned long long bytes) -> long long {      // block-uniform result; -1: does not fit now, -2: can never fit
        if (c.tid() == 0) { long long r; bytes = (bytes + 255ULL) & ~255ULL;
            if (bytes > spool_cap) r = -2; else { unsigned long long at = atomic_add64(&bc->s1_pool_used, bytes); r = at + bytes <= spool_cap ? (long long)at : -1; }
            sh.bcast64[2] = r; }
        c.sync(); long long r = sh.bcast64[2]; c.sync(); return r;
    };
    auto give_up = [&](long long why) { clear_bits(); if (c.tid() == 0) { rec.state = why == -2 ? -1 : 2; rec.n_cand = n_cand; rec.K = p.depth; rec.path = path; if (why != -2) atomic_add(&bc->s1_deferred, 1); else out.n[0] = -1; } c.sync(); };      // a query larger than the whole pool is an overflow, like every other fixed buffer
    const long long a1 = pool_alloc(8ULL * (unsigned long long)n_cand + 64);
    if (a1 < 0) { give_up(a1); return; }
    int32_t* cand = reinterpret_cast<int32_t*>(spool + a1); float* dlp = reinterpret_cast<float*>(spool + a1 + (((long long)n_cand * 4 + 31) & ~31LL));
    // ---- 1b. expand + candidates before every container
    {   int run = wbase;
        for (int64_t gb = w0; gb < w1; gb += 4 * WS) {          // four groups per trip: their words are loaded together, then scanned one after the other
            unsigned vv[4];
            for (int u = 0; u < 4; u++) { const int64_t g = gb + u * WS, w = g + c.lane(); vv[u] = (g < w1 && sh.dirty[g >> 11] && w < w1) ? ws.bits[w] : 0u; }
            for (int u = 0; u < 4; u++) {
                const int64_t g0 = gb + u * WS; if (g0 >= w1) break;
                if (!sh.dirty[g0 >> 11]) { if ((g0 & 2047) == 0 && c.lane() == 0) ws.cstart[g0 >> 11] = run; continue; }
                const int64_t w = g0 + c.lane(); unsigned v = vv[u]; const int pc = popc(v); int incl = pc;
                for (int d = 1; d < WS; d <<= 1) { int o = c.shfl(incl, c.lane() >= d ? c.lane() - d : 0); if (c.lane() >= d) incl += o; }
                int o = run + incl - pc;
                if (w < w1 && (w & 2047) == 0) ws.cstart[w >> 11] = o;
                while (v) { int b = ffs32(v) - 1; v &= v - 1; cand[o++] = (int32_t)((w << 5) | b); }
                run += c.shfl(incl, WS - 1);
            }
        }
        if (c.tid() == 0) ws.cstart[ncont] = n_cand;
    }
    c.sync();
    IFX_LTICK(0);   // count + expand
    // ---- 2. lengths, deleted flags (folded into the id), chunk table
    const bool any_deleted = ix.n_live != ix.n_docs;
    for (int i0 = c.tid(); i0 < n_cand; i0 += 8 * NT) {
        int d[8]; float dl[8]; uint8_t del[8];
        for (int u = 0; u < 8; u++) { int i = i0 + u * NT; d[u] = i < n_cand ? cand[i] : -1; }
        for (int u = 0; u < 8; u++) if (d[u] >= 0) { dl[u] = ix.doc_len[d[u]]; del[u] = any_deleted ? ix.deleted[d[u]] : (uint8_t)0; }
        for (int u = 0; u < 8; u++) if (d[u] >= 0) { int i = i0 + u * NT; dlp[i] = dl[u]; if (del[u]) cand[i] = d[u] | DEL_BIT; }
    }
    IFX_LTICK(1);   // document lengths + deleted flags
    int Ta = 0;
    if (c.tid() == 0) { for (int t = 0; t < T; t++) sh.order[t] = sh.terms[t].idf > 0.f ? Ta++ : -1; sh.bcast[0] = Ta; sh.bcast[1] = 0; sh.bcast[2] = 0; sh.bcast[3] = 0; }   // sh.order: term -> row of the tf matrix
    c.sync();
    Ta = sh.bcast[0];
    int n_chunks = 0, n_slots = 0;      // running totals: chunks, padded slots
    for (int c0 = 0; c0 < ncont; c0 += NT) {
        const int cc = c0 + c.tid(); const int cntc = cc < ncont ? ws.cstart[cc + 1] - ws.cstart[cc] : 0;
        const int nch = (cntc + CHUNK - 1) / CHUNK; const int slots = (cntc / CHUNK) * CHUNK + pad16(cntc % CHUNK);
        int t1, t2; const int e1 = block_excl_scan(c, nch, sh.scan, t1); const int e2 = block_excl_scan(c, slots, sh.scan, t2);
        if (cc < ncont) { ws.cfirst[cc] = n_chunks + e1;
                          S1Cont ct; ct.cstart = ws.cstart[cc]; ct.cnt = cntc; ct.cpad = n_slots + e2; ct.cfirst = n_chunks + e1; reinterpret_cast<S1Cont*>(ws.ctab)[cc] = ct; }
        if (cntc > 0) atomic_max(&sh.bcast[1], cntc < CHUNK ? cntc : CHUNK);
        n_chunks += t1; n_slots += t2;
    }
    c.sync();
    const int max_cnt = sh.bcast[1]; const S1Cont* ctab = reinterpret_cast<const S1Cont*>(ws.ctab);
    const unsigned long long tf_bytes = (unsigned long long)(Ta > 0 ? Ta : 1) * (unsigned long long)n_slots;
    const unsigned long long chunk_bytes = ((unsigned long long)n_chunks * sizeof(S1Chunk) + 15ULL) & ~15ULL, term_bytes = (unsigned long long)(Ta > 0 ? Ta : 1) * sizeof(S1TermP);
    const long long a2 = pool_alloc(chunk_bytes + term_bytes + tf_bytes + 64);
    if (a2 < 0) { give_up(a2); return; }
    S1Chunk* chunks = reinterpret_cast<S1Chunk*>(spool + a2); S1TermP* tparams = reinterpret_cast<S1TermP*>(spool + a2 + chunk_bytes);
    uint8_t* tfb = spool + a2 + chunk_bytes + term_bytes;
    for (int cc = c.tid(); cc < ncont; cc += NT) {
        const int cntc = ws.cstart[cc + 1] - ws.cstart[cc]; const int nch = (cntc + CHUNK - 1) / CHUNK;
        for (int s = 0; s < nch; s++) { S1Chunk ch; ch.start = ws.cstart[cc] + s * CHUNK; ch.cnt = cntc - s * CHUNK < CHUNK ? cntc - s * CHUNK : CHUNK; ch.tf_off = (int64_t)Ta * (ctab[cc].cpad + s * CHUNK); chunks[ws.cfirst[cc] + s] = ch; }
    }
    for (int t = c.tid(); t < T; t += NT) if (sh.order[t] >= 0) { S1TermP tp; tp.idf = sh.terms[t].idf; tp.max_score = sh.terms[t].max_score; tp.suffix_after = sh.terms[t].suffix_after; tp.pad = 0; tparams[sh.order[t]] = tp; }
    {   // zero the tf matrix (16-byte stores; the block is 16-byte aligned and padded)
        struct alignas(16) Z16 { unsigned v[4]; }; Z16 z; z.v[0] = z.v[1] = z.v[2] = z.v[3] = 0u; Z16* zp = reinterpret_cast<Z16*>(tfb);
        for (unsigned long long i = c.tid(); i < (tf_bytes + 15ULL) / 16ULL; i += NT) zp[i] = z;
    }
    c.sync();
    IFX_LTICK(2);   // chunk table + zeroed tf matrix
    // ---- 3. tf lookups
    unsigned long long cost_s = 0; int n_dict = 0;
    for (int t = 0; t < T; t++) if (sh.order[t] >= 0 && sh.terms[t].term_id >= 0) { cost_s += 5ULL * (unsigned long long)sh.terms[t].len; n_dict++; }
    const bool forward = force_mode == 1 ? true : (force_mode == 2 ? false : (n_dict > 0 && 3ULL * (unsigned long long)n_cand * (unsigned long long)fwd_avg_bytes < cost_s));      // random forward-list reads cost ~3x a streamed byte (measured, profiles/r2)
    if (forward) {
        // Batches of FW_G candidates per warp: their forward lists (a few dozen to a few hundred (term, tf) pairs each) are walked as ONE
        // concatenated range, so a lane has several independent loads in flight instead of one dependent chain per candidate. The
        // query's term hash maps term id -> row.
        constexpr int FW_G = Ctx::WS >= 4 ? 4 : 1;      // (the single-lane test build walks one candidate at a time)
        for (int k = 0; k < n_chunks; k++) {
            const S1Chunk ch = chunks[k]; const int rowlen = pad16(ch.cnt);
            for (int jb = c.warp() * FW_G; jb < ch.cnt; jb += NW * FW_G) {
                int64_t r0 = 0, r1 = 0;
                if (c.lane() < FW_G && jb + c.lane() < ch.cnt) { const int d = cand[ch.start + jb + c.lane()] & ~DEL_BIT; r0 = ix.fwd_ptr[d]; r1 = ix.fwd_ptr[d + 1]; }
                int64_t b0[FW_G]; int pre[FW_G + 1]; pre[0] = 0;
                for (int g = 0; g < FW_G; g++) { b0[g] = c.shfl(r0, g); const int64_t e1 = c.shfl(r1, g); pre[g + 1] = pre[g] + (int)(e1 - b0[g]); }
                const int E = pre[FW_G];
                for (int e0 = c.lane(); e0 < E; e0 += 4 * WS) {
                    int32_t tid[4]; uint8_t tfv[4]; int gj[4];
                    for (int u = 0; u < 4; u++) { const int e = e0 + u * WS; tid[u] = -1; gj[u] = 0; if (e < E) { int g = 0; for (int x = 1; x < FW_G; x++) if (e >= pre[x]) g = x; const int64_t i = b0[g] + (e - pre[g]); tid[u] = ix.fwd_term[i]; tfv[u] = ix.fwd_tf[i]; gj[u] = g; } }
                    for (int u = 0; u < 4; u++) if (tid[u] >= 0) { unsigned h = qh_hash(tid[u]);
                        for (;;) { const int32_t kk = sh.qh_key[h]; if (kk == tid[u]) { tfb[ch.tf_off + (int64_t)sh.order[sh.qh_slot[h]] * rowlen + jb + gj[u]] = tfv[u]; break; } if (kk < 0) break; h = (h + 1) & (QH_SIZE - 1); } }
                }
            }
        }
        c.sync();
        IFX_LTICK(3);   // forward-index lookups
    }
    // Streamed lists: every scored list, or in forward mode the LD1 unions (they have no term id, hence no forward entries).
    if (c.tid() == 0) { int ns = 0; for (int t = 0; t < T; t++) if (sh.order[t] >= 0 && (!forward || sh.terms[t].term_id < 0)) { sh.slist[ns] = (uint8_t)t; sh.srow[ns] = (uint8_t)sh.order[t]; ns++; } sh.bcast[2] = ns; }
    c.sync();
    const int Ts = sh.bcast[2];
    if (Ts > 0) {
        // Where each list enters every container: ws.lrange[j][cc], one thread per (list, container) pair. Long dictionary lists read
        // their skip table; short ones and the LD1 unions (sorted, no skip table) are searched, once per query rather than once per
        // container inside the loop below. Only the bounds of containers with candidates are needed.
        const int NC1 = ncont + 1;
        for (int i = c.tid(); i < Ts * NC1; i += NT) {
            const int j = i / NC1, cc = i - j * NC1;
            if (!((cc < ncont && sh.dirty[cc]) || (cc > 0 && sh.dirty[cc - 1]))) continue;
            const TermS& tm = sh.terms[sh.slist[j]];
            ws.lrange[i] = tm.skip ? tm.skip[cc] : (int32_t)lower_bound_i32(tm.docs, 0, tm.len, cc << 16);
        }
        c.sync();
        IFX_LTICK(5);   // per-container list ranges
        // Container-major lookups: the container's bitset words and their candidate ranks go to shared memory; then the container's
        // postings of all streamed lists, concatenated into one range, are spread over the whole block. A list's part of the range
        // starts at the 16-byte boundary before its first posting and is padded to whole groups of four, so that a group lies in one
        // list and, when all four are its postings, is one 16-byte id load plus one 4-byte tf load; LG groups per thread in flight.
        // A hit's slot follows from the rank within the container and the container's sub-chunk layout.
        constexpr int LG = 4;
        struct alignas(16) Id4 { int32_t v[4]; };
        for (int cc = 0; cc < ncont; cc++) {
            if (!sh.dirty[cc]) continue;                  // (uniform) never touched: no candidates
            const S1Cont ct = ctab[cc];
            if (ct.cnt == 0) continue;
            const unsigned* bw = ws.bits + (int64_t)cc * CONT_WORDS;      // (the bitset is allocated to whole containers)
            for (int w = c.tid(); w < CONT_WORDS; w += NT) sh.cbits[w] = bw[w];
            for (int j = c.tid(); j < Ts; j += NT) {
                const TermS& tm = sh.terms[sh.slist[j]]; const int32_t r0 = ws.lrange[j * NC1 + cc], n = ws.lrange[j * NC1 + cc + 1] - r0;
                const int32_t* dp = tm.docs + r0; const int m = (int)((reinterpret_cast<uintptr_t>(dp) >> 2) & 3);
                sh.sdoc[j] = dp - m; sh.stf[j] = tm.tf ? tm.tf + r0 - m : nullptr; sh.smis[j] = (uint8_t)m; sh.slen[j] = n > 0 ? m + n : 0;
            }
            c.sync();
            {   // exclusive candidate rank of every word: each thread owns `per` consecutive words
                const int per = (CONT_WORDS + NT - 1) / NT, w0 = c.tid() * per; int mine = 0, tot;
                for (int k = 0; k < per && w0 + k < CONT_WORDS; k++) mine += popc(sh.cbits[w0 + k]);
                int r = block_excl_scan(c, mine, sh.scan, tot);
                for (int k = 0; k < per && w0 + k < CONT_WORDS; k++) { sh.crank[w0 + k] = (uint16_t)r; r += popc(sh.cbits[w0 + k]); }
            }
            {   // start of every list's padded part in the concatenated range
                const int per = (Ts + NT - 1) / NT, j0 = c.tid() * per; int mine = 0, E;
                for (int k = 0; k < per && j0 + k < Ts; k++) mine += (sh.slen[j0 + k] + 3) & ~3;
                int r = block_excl_scan(c, mine, sh.scan, E);
                for (int k = 0; k < per && j0 + k < Ts; k++) { sh.spre[j0 + k] = r; r += (sh.slen[j0 + k] + 3) & ~3; }
                if (c.tid() == 0) sh.spre[Ts] = E;
            }
            c.sync();
            const int G = sh.spre[Ts] >> 2; int j = 0;
            for (int g0 = c.tid(); g0 < G; g0 += LG * NT) {
                Id4 dv[LG]; unsigned tw[LG]; const int jr = j;      // a group's docs (-1: not a posting of the list) and tfs; the list index at the first group
#pragma unroll
                for (int u = 0; u < LG; u++) {
                    const int g = g0 + u * NT; tw[u] = 0u;
#pragma unroll
                    for (int x = 0; x < 4; x++) dv[u].v[x] = -1;
                    if (g < G) {
                        while (4 * g >= sh.spre[j + 1]) j++;      // (groups of a thread ascend: the list index only moves forward)
                        const int k = 4 * g - sh.spre[j], lo = sh.smis[j], hi = sh.slen[j]; const int32_t* dp = sh.sdoc[j] + k; const uint8_t* tp = sh.stf[j];
                        if (k >= lo && k + 4 <= hi) { dv[u] = *reinterpret_cast<const Id4*>(dp); tw[u] = tp ? *reinterpret_cast<const unsigned*>(tp + k) : 0x01010101u; }
                        else {
#pragma unroll
                            for (int x = 0; x < 4; x++) if (k + x >= lo && k + x < hi) { dv[u].v[x] = dp[x]; tw[u] |= (tp ? (unsigned)tp[k + x] : 1u) << (8 * x); }
                        }
                    }
                }
                j = jr;      // walked again for the rows: cheaper than holding them across the loads
#pragma unroll
                for (int u = 0; u < LG; u++) {
                    const int g = g0 + u * NT; if (g >= G) break;
                    while (4 * g >= sh.spre[j + 1]) j++;
                    const int64_t row = sh.srow[j];
#pragma unroll
                    for (int x = 0; x < 4; x++) {
                        const int d = dv[u].v[x]; if (d < 0) continue;
                        const int w = (d >> 5) & (CONT_WORDS - 1); const unsigned bits = sh.cbits[w], bit = 1u << (d & 31);
                        if (bits & bit) {
                            const int jc = sh.crank[w] + popc(bits & (bit - 1)), sub = jc / CHUNK; const int cnt_k = ct.cnt - sub * CHUNK < CHUNK ? ct.cnt - sub * CHUNK : CHUNK;
                            tfb[(int64_t)Ta * (ct.cpad + sub * CHUNK) + row * pad16(cnt_k) + (jc - sub * CHUNK)] = (uint8_t)(tw[u] >> (8 * x));
                        }
                    }
                }
            }
            c.sync();                                     // the slice is rewritten for the next container
        }
        IFX_LTICK(6);   // container-major streamed lookups
    }
    // ---- 4. bitset back to all-zero; record, queue, roofline accounting (SURVEY 8d)
    clear_bits();
    IFX_LTICK(4);   // bitset cleared
    if (c.tid() == 0) {
        rec.off_cand = a1; rec.off_dl = a1 + (((long long)n_cand * 4 + 31) & ~31LL); rec.off_chunk = a2; rec.off_terms = a2 + (long long)chunk_bytes; rec.off_tf = a2 + (long long)(chunk_bytes + term_bytes);
        rec.n_cand = n_cand; rec.n_chunks = n_chunks; rec.n_terms = Ta; rec.max_cnt = max_cnt; rec.K = p.depth; rec.path = path;
        const bool warp_ok = Ta <= W_TERMS && p.depth <= W_K;
        if (Ta == 0) rec.state = 0;
        else if (warp_ok && max_cnt <= W_CAP) { rec.state = 1; queues.light[atomic_add(&bc->s1_n_light, 1)] = q; }
        else if (warp_ok && max_cnt <= W_CAP_MID) { rec.state = 4; queues.mid[atomic_add(&bc->s1_n_mid, 1)] = q; }
        else { rec.state = 3; queues.heavy[atomic_add(&bc->s1_n_heavy, 1)] = q; }
        unsigned long long algo = path == 1 ? 4ULL * (unsigned long long)n_cand : 2ULL * (unsigned long long)((ix.n_docs + 7) / 8);
        for (int i = 0; i < T; i++) {
            unsigned long long full = (sh.terms[i].tf ? 5ULL : 4ULL) * (unsigned long long)sh.terms[i].len;
            bool streamed = (sh.streamed_mask[i >> 6] >> (i & 63)) & 1ULL; unsigned long long probe = 32ULL * (unsigned long long)n_cand;
            algo += streamed ? full : (full < probe ? full : probe);
        }
        algo += 4ULL * (unsigned long long)n_cand;
        atomic_add64(&bc->algo_bytes, algo); atomic_add64(&bc->s1_cand_sum, (unsigned long long)n_cand);
        if (out.dbg) { out.dbg[0] = n_cand; out.dbg[6] = forward ? 1 : 2; out.dbg[7] = n_chunks; out.dbg[8] = max_cnt; out.dbg[9] = Ta; }
    }
    c.sync();
}

// ---------------------------------------------------------------------------------------------------------------
// score_warp: one warp scores one light query. Slot j of a chunk lives in lane j % 32, register j / 32 (candidate order = slot order),
// so ranks come from ballots; nothing leaves the warp. Same arithmetic, the same order of operations and the same heap replay as the
// block-wide scorer below.
struct WarpScoreShared {
    alignas(16) float heap_pr[W_K + 8]; int32_t heap_doc[W_K + 8];
    alignas(16) uint8_t tf[W_TF];                 // a tile of the current chunk's tf rows; reused for the flush survivors ((doc, score) pairs)
    S1TermP terms[W_TERMS];
};

// CAPW: slot capacity of a chunk (W_CAP or W_CAP_MID); lane l owns slots l, l + 32, ... (CAPW / 32 registers each for score and length)
template <int CAPW>
IFX_FN void score_warp(const Ctx& c, float avgdl_in, const S1Rec& rec, const unsigned char* spool, WarpScoreShared& sh, int32_t* out_doc, float* out_score, int32_t* out_n) {
    constexpr int WS = Ctx::WS; constexpr int W_R = CAPW / WS; const int lane = c.lane();
    const int K = rec.K, Ta = rec.n_terms; const float avgdl = avgdl_in > 0.f ? avgdl_in : 1.f;
    const int32_t* cand = reinterpret_cast<const int32_t*>(spool + rec.off_cand); const float* dlp = reinterpret_cast<const float*>(spool + rec.off_dl);
    const S1Chunk* chunks = reinterpret_cast<const S1Chunk*>(spool + rec.off_chunk); const S1TermP* tparams = reinterpret_cast<const S1TermP*>(spool + rec.off_terms);
    const uint8_t* tfb = spool + rec.off_tf;
    for (int i = lane; i < W_K + 8; i += WS) { sh.heap_pr[i] = 3.0e38f; sh.heap_doc[i] = 0; }
    for (int i = lane; i < Ta; i += WS) sh.terms[i] = tparams[i];
    c.syncwarp();
    float thr = 0.f; int hs = 0;
    for (int k = 0; k < rec.n_chunks; k++) {
        const S1Chunk ch = chunks[k]; const int cnt = ch.cnt, rowlen = pad16(cnt); const int rows_per_tile = W_TF / rowlen < Ta ? W_TF / rowlen : Ta;
        float sc[W_R], nv[W_R];      // score and the length norm of the Vector256 form (one evaluation per slot and chunk; the scalar form re-reads the length)
#pragma unroll
        for (int r = 0; r < W_R; r++) { const int j = r * WS + lane; sc[r] = 0.f; nv[r] = j < cnt ? bm25_norm_vector(dlp[ch.start + j], avgdl) : 0.f; }
        for (int a0 = 0; a0 < Ta; a0 += rows_per_tile) {
            const int tile = Ta - a0 < rows_per_tile ? Ta - a0 : rows_per_tile;
            {   // the tile's rows: contiguous in the chunk's block, 16-byte aligned
                struct alignas(16) V16 { unsigned v[4]; }; const V16* src = reinterpret_cast<const V16*>(tfb + ch.tf_off + (int64_t)a0 * rowlen); V16* dst = reinterpret_cast<V16*>(sh.tf); const int n16 = tile * rowlen / 16;
                c.syncwarp();
                for (int i = lane; i < n16; i += WS) dst[i] = src[i];
                c.syncwarp();
            }
            for (int a = a0; a < a0 + tile; a++) {
                const S1TermP tp = sh.terms[a]; const uint8_t* row = sh.tf + (a - a0) * rowlen;
                const bool uns = !((0.f + tp.max_score) + tp.suffix_after <= thr);      // the test cannot fire for any score >= 0 (float addition is monotone): every non-zero tf is a match
                int m = 0;
#pragma unroll
                for (int r = 0; r < W_R; r++) {      // MaxScore test (Bm25Scorer.cs:354): matches of this term in the chunk
                    const int j = r * WS + lane; const unsigned tfv = j < cnt ? row[j] : 0u;
                    m += popc(c.ballot(tfv != 0u && (uns || !(sc[r] + tp.max_score + tp.suffix_after <= thr))));
                }
                if (m == 0) continue;
                const int vec_end = m - (m & 7); int run = 0;
#pragma unroll
                for (int r = 0; r < W_R; r++) {      // rank among them (candidate order = slot order) selects the Vector256 or the scalar form
                    const int j = r * WS + lane; const unsigned tfv = j < cnt ? row[j] : 0u;
                    const bool al = tfv != 0u && (uns || !(sc[r] + tp.max_score + tp.suffix_after <= thr));
                    const unsigned bm = c.ballot(al);
                    if (al) { const int rank = run + popc(bm & c.lanemask_lt()); const float tf = (float)tfv;
                        sc[r] += rank < vec_end ? bm25_from_norm_vector(tf, nv[r], tp.idf) : bm25_scalar(tf, dlp[ch.start + j], avgdl, tp.idf); }
                    run += popc(bm);
                }
            }
        }
        c.syncwarp();
        // flush (Bm25Scorer.cs:316-329): eligibility against the chunk-start threshold, survivors in candidate order, then the exact heap replay
        // (the survivor buffer holds W_TF / 8 pairs: larger sets are drained in rounds, order preserved)
        unsigned long long* surv = reinterpret_cast<unsigned long long*>(sh.tf); const bool full = hs >= K; const float thr0 = thr; constexpr int SCAP = W_TF / 8;
        for (int r0 = 0; r0 < W_R; r0 += SCAP / WS) {
            int ns = 0;
#pragma unroll
            for (int rr = 0; rr < SCAP / WS; rr++) { const int r = r0 + rr; if (r >= W_R) break;
                const int j = r * WS + lane; const bool e0 = j < cnt && sc[r] > 0.f && (!full || sc[r] > thr0);
                int id = e0 ? cand[ch.start + j] : DEL_BIT; const bool e = e0 && id >= 0;      // deleted documents carry bit 31
                const unsigned bm = c.ballot(e); if (e) surv[ns + popc(bm & c.lanemask_lt())] = kv_pack(id, sc[r]); ns += popc(bm);
            }
            c.syncwarp();
            if (lane == 0) {
                for (int i = 0; i < ns; i++) { const unsigned long long kv = surv[i]; const float s = kv_score(kv);
                    if (hs < K) { heap_move_up(sh, (int)(kv >> 32), s, hs); hs++; if (hs == K) thr = sh.heap_pr[3]; }
                    else if (s > thr) thr = heap_replace_root(sh, (int)(kv >> 32), s, hs); }
            }
            thr = c.shfl(thr, 0); hs = c.shfl(hs, 0);
            c.syncwarp();
        }
    }
    for (int i = lane; i < hs; i += WS) { out_doc[i] = sh.heap_doc[i + 3]; out_score[i] = sh.heap_pr[i + 3]; }
    if (lane == 0) out_n[0] = hs;
    c.syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// score_cta: one CTA scores one heavy query (chunks of up to 4096 candidates). Warp 0 replays the heap over the previous chunk's
// survivors while warps 1.. copy the next chunk's block into shared memory; phase B (MaxScore test, rank -> Vector256 / scalar form,
// accumulation) runs tile by tile over 6 terms, every thread owning 8 consecutive slots.
IFX_FN void score_cta(const Ctx& c, float avgdl_in, const S1Rec& rec, const unsigned char* spool, S1Workspace& ws, S1Shared& sh, int32_t* out_doc, float* out_score, int32_t* out_n) {
    const int K = rec.K, T = rec.n_terms, NT = c.nthreads(), NW = c.nwarps(); const float avgdl = avgdl_in > 0.f ? avgdl_in : 1.f;
    const int32_t* cand = reinterpret_cast<const int32_t*>(spool + rec.off_cand); const float* dlp = reinterpret_cast<const float*>(spool + rec.off_dl);
    const S1Chunk* chunks = reinterpret_cast<const S1Chunk*>(spool + rec.off_chunk); const S1TermP* tparams = reinterpret_cast<const S1TermP*>(spool + rec.off_terms);
    const uint8_t* tfb = spool + rec.off_tf;
    for (int i = c.tid(); i < MAX_K + 8; i += NT) { sh.heap_pr[i] = 3.0e38f; sh.heap_doc[i] = 0; }
    for (int i = c.tid(); i < T; i += NT) { const S1TermP tp = tparams[i]; sh.terms[i].idf = tp.idf; sh.terms[i].max_score = tp.max_score; sh.terms[i].suffix_after = tp.suffix_after; }
    if (c.tid() == 0) { sh.heap_size = 0; sh.thr = 0.f; }
    c.sync();
    const int hw = NT > Ctx::WS ? Ctx::WS : 0; const bool worker = c.tid() >= hw; const int wt = c.tid() - hw, NTW = NT - hw;
    int pend = 0;
    auto drain = [&]() {                                       // Bm25Scorer.cs:316-329 + UpdateTopK (:654-670) over the compacted survivors, in candidate order
        float thr_r = sh.thr; int hs = sh.heap_size;
        auto one = [&](unsigned long long kv) { const float s = kv_score(kv);
            if (hs < K) { heap_move_up(sh, (int)(kv >> 32), s, hs); hs++; if (hs == K) thr_r = sh.IFX_HP(0); }
            else if (s > thr_r) thr_r = heap_replace_root(sh, (int)(kv >> 32), s, hs); };
        if (pend <= SURV_CAP) { for (int i = 0; i < pend; i++) one(sh.surv[i]); }
        else for (int i = 0; i < pend; i += 8) { unsigned long long kv[8]; for (int u = 0; u < 8; u++) kv[u] = i + u < pend ? ws.surv_g[i + u] : 0ULL; for (int u = 0; u < 8; u++) if (i + u < pend) one(kv[u]); }
        sh.thr = thr_r; sh.heap_size = hs;
    };
    auto copy_rows = [&](const S1Chunk& ch, int t0, int tile, int me, int nme) {       // rows t0 .. t0+tile of the chunk's tf block -> sh.tfm
        struct alignas(16) V16 { unsigned v[4]; }; const int rowlen = pad16(ch.cnt), n16 = rowlen / 16;
        for (int i = me; i < tile * n16; i += nme) { const int tt = i / n16, x = i - tt * n16; reinterpret_cast<V16*>(sh.tfm[tt])[x] = reinterpret_cast<const V16*>(tfb + ch.tf_off + (int64_t)(t0 + tt) * rowlen)[x]; }
    };
    for (int k = 0; k < rec.n_chunks; k++) {
        const S1Chunk ch = chunks[k]; const int cnt = ch.cnt;
        if (c.tid() == 0 && pend) drain();
        if (worker) {
            for (int j = wt; j < cnt; j += NTW) { sh.cand_s[j] = cand[ch.start + j]; sh.nv_s[j] = bm25_norm_vector(dlp[ch.start + j], avgdl); sh.score[j] = 0.f; }
            copy_rows(ch, 0, T < S1_TILE ? T : S1_TILE, wt, NTW);
        }
        c.sync();      // join: heap drained, chunk staged, tile 0 copied
        const float thr = sh.thr; const int rounds = (cnt + NT - 1) / NT;
        const int per_thread = (CHUNK + NT - 1) / NT; const int j0 = c.tid() * per_thread < cnt ? c.tid() * per_thread : cnt; const int j1 = j0 + per_thread < cnt ? j0 + per_thread : cnt;
        for (int t0 = 0; t0 < T; t0 += S1_TILE) {
            const int tile = T - t0 < S1_TILE ? T - t0 : S1_TILE;
            if (t0 > 0) { copy_rows(ch, t0, tile, c.tid(), NT); c.sync(); }
            int nscan = 0;
#ifndef IFX_EMU
            const bool fast = per_thread == 8 && j1 - j0 == 8;      // the 8 owned slots live in registers for the whole term
            // A term whose own bound plus the bounds of the terms after it already exceeds the threshold can never be skipped (scores are
            // >= 0 and float addition is monotone), so its matches are exactly the non-zero tf slots: the ranks of all such terms of the
            // tile come from ONE packed block scan (16-bit fields, <= 4096 each).
            unsigned uns = 0, ex01 = 0, ex23 = 0, ex45 = 0, m01 = 0, m23 = 0, m45 = 0;
            {   bool u = false; if (c.lane() < tile) { const TermS& tm = sh.terms[t0 + c.lane()]; u = !((0.f + tm.max_score) + tm.suffix_after <= thr); }
                uns = __ballot_sync(0xffffffffu, u); }
            if (__popc(uns) >= 2) {
                unsigned pk[3] = {0u, 0u, 0u};
#pragma unroll
                for (int tt = 0; tt < S1_TILE; tt++) if ((uns >> tt) & 1u) {
                    const uint8_t* tfr = sh.tfm[tt]; unsigned n = 0;
                    if (fast) { unsigned long long v = *reinterpret_cast<const unsigned long long*>(tfr + j0); v |= v >> 4; v |= v >> 2; v |= v >> 1; n = (unsigned)__popcll(v & 0x0101010101010101ULL); }
                    else for (int j = j0; j < j1; j++) n += tfr[j] != 0;
                    pk[tt >> 1] |= n << (16 * (tt & 1));
                }
                unsigned in0 = pk[0], in1 = pk[1], in2 = pk[2];
                for (int d = 1; d < 32; d <<= 1) {
                    unsigned o0 = __shfl_up_sync(0xffffffffu, in0, d), o1 = __shfl_up_sync(0xffffffffu, in1, d), o2 = __shfl_up_sync(0xffffffffu, in2, d);
                    if (c.lane() >= d) { in0 += o0; in1 += o1; in2 += o2; }
                }
                if (c.lane() == 31) { sh.scan3[c.warp()][0] = in0; sh.scan3[c.warp()][1] = in1; sh.scan3[c.warp()][2] = in2; }
                c.sync();
                uint4 x = make_uint4(0u, 0u, 0u, 0u); if (c.lane() < NW) x = *reinterpret_cast<const uint4*>(sh.scan3[c.lane()]);
                for (int d = 1; d < NW; d <<= 1) {
                    unsigned o0 = __shfl_up_sync(0xffffffffu, x.x, d), o1 = __shfl_up_sync(0xffffffffu, x.y, d), o2 = __shfl_up_sync(0xffffffffu, x.z, d);
                    if (c.lane() >= d) { x.x += o0; x.y += o1; x.z += o2; }
                }
                const int src = c.warp() > 0 ? c.warp() - 1 : 0;
                unsigned b0 = __shfl_sync(0xffffffffu, x.x, src), b1 = __shfl_sync(0xffffffffu, x.y, src), b2 = __shfl_sync(0xffffffffu, x.z, src);
                if (c.warp() == 0) { b0 = 0; b1 = 0; b2 = 0; }
                m01 = __shfl_sync(0xffffffffu, x.x, NW - 1); m23 = __shfl_sync(0xffffffffu, x.y, NW - 1); m45 = __shfl_sync(0xffffffffu, x.z, NW - 1);
                ex01 = b0 + in0 - pk[0]; ex23 = b1 + in1 - pk[1]; ex45 = b2 + in2 - pk[2];
            } else uns = 0;
#else
            const bool fast = false; const unsigned uns = 0;
#endif
            for (int tt = 0; tt < tile; tt++) {
                const TermS& tm = sh.terms[t0 + tt]; const uint8_t* tfr = sh.tfm[tt];
                int mine = 0; const float tbound = tm.max_score; const float tsuffix = tm.suffix_after;
                const bool ranked = (uns >> tt) & 1u;              // uniform: rank and match count already known, every non-zero tf is a match
#ifndef IFX_EMU
                unsigned long long tf8 = 0ULL; unsigned alive = 0; float sc8[8];
                if (fast) {
                    tf8 = *reinterpret_cast<const unsigned long long*>(tfr + j0);
                    if (tf8 != 0ULL) {
                        float4 sa = *reinterpret_cast<const float4*>(&sh.score[j0]), sb = *reinterpret_cast<const float4*>(&sh.score[j0 + 4]);
                        sc8[0] = sa.x; sc8[1] = sa.y; sc8[2] = sa.z; sc8[3] = sa.w; sc8[4] = sb.x; sc8[5] = sb.y; sc8[6] = sb.z; sc8[7] = sb.w;
#pragma unroll
                        for (int kk = 0; kk < 8; kk++) { unsigned tfv = (unsigned)(tf8 >> (8 * kk)) & 0xFFu; if (tfv != 0 && (ranked || !(sc8[kk] + tbound + tsuffix <= thr))) alive |= 1u << kk; }
                        mine = __popc(alive);
                    }
                } else
#endif
                { for (int j = j0; j < j1; j++) if (tfr[j] != 0 && (ranked || !(sh.score[j] + tbound + tsuffix <= thr))) mine++; }
                int m, rank;
#ifndef IFX_EMU
                if (ranked) { const unsigned e = tt < 2 ? ex01 : (tt < 4 ? ex23 : ex45), tm_ = tt < 2 ? m01 : (tt < 4 ? m23 : m45); rank = (int)((e >> (16 * (tt & 1))) & 0xFFFFu); m = (int)((tm_ >> (16 * (tt & 1))) & 0xFFFFu); }
                else
#endif
                { rank = block_excl_scan_1b(c, mine, sh.scan2[nscan & 1], m); nscan++; }
                const int vec_end = m - (m & 7);
#ifndef IFX_EMU
                if (fast) {
                    if (alive) {
                        float4 da = *reinterpret_cast<const float4*>(&sh.nv_s[j0]), db = *reinterpret_cast<const float4*>(&sh.nv_s[j0 + 4]);
                        float nv8[8] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
#pragma unroll
                        for (int kk = 0; kk < 8; kk++) if (alive & (1u << kk)) {
                            float tf = (float)((unsigned)(tf8 >> (8 * kk)) & 0xFFu);
                            float add = rank < vec_end ? bm25_from_norm_vector(tf, nv8[kk], tm.idf) : bm25_scalar(tf, dlp[ch.start + j0 + kk], avgdl, tm.idf);
                            sc8[kk] += add; rank++;
                        }
                        *reinterpret_cast<float4*>(&sh.score[j0]) = make_float4(sc8[0], sc8[1], sc8[2], sc8[3]);
                        *reinterpret_cast<float4*>(&sh.score[j0 + 4]) = make_float4(sc8[4], sc8[5], sc8[6], sc8[7]);
                    }
                } else
#endif
                for (int j = j0; j < j1; j++) {
                    const uint8_t tfv = tfr[j];
                    if (tfv != 0 && (ranked || !(sh.score[j] + tbound + tsuffix <= thr))) {
                        float tf = (float)tfv;
                        float s2 = rank < vec_end ? bm25_from_norm_vector(tf, sh.nv_s[j], tm.idf) : bm25_scalar(tf, dlp[ch.start + j], avgdl, tm.idf);
                        sh.score[j] += s2; rank++;
                    }
                }
                // no further barrier: score[j] of these slots is private to this thread throughout the tile
            }
            c.sync();                                    // the tile buffer is rewritten by arbitrary threads for the next tile / chunk
        }
        {   // flush, part 1: eligibility in parallel against the chunk-start threshold, survivors compacted in candidate order (part 2 = drain)
            const bool full = sh.heap_size >= K;
            for (int r = 0; r < rounds; r++) {
                int j = r * NT + c.tid();
                bool e = j < cnt && sh.score[j] > 0.f && (!full || sh.score[j] > thr) && sh.cand_s[j] >= 0;      // deleted documents carry bit 31
                unsigned b = c.ballot(e);
                if (c.lane() == 0) sh.ballots[0][r * NW + c.warp()] = b;
            }
            c.sync();
            const int slots = rounds * NW;
            if (c.warp() == 0) {     // exclusive prefix of the ballot popcounts (slot order == candidate order)
                int per = (slots + Ctx::WS - 1) / Ctx::WS; int s0 = c.lane() * per < slots ? c.lane() * per : slots, s1 = s0 + per < slots ? s0 + per : slots; int mine = 0;
                for (int sl = s0; sl < s1; sl++) mine += popc(sh.ballots[0][sl]);
                int incl = mine;
                for (int d = 1; d < Ctx::WS; d <<= 1) { int o = c.shfl(incl, c.lane() >= d ? c.lane() - d : 0); if (c.lane() >= d) incl += o; }
                int run = incl - mine;
                for (int sl = s0; sl < s1; sl++) { sh.bprefix[sl] = run; run += popc(sh.ballots[0][sl]); }
                if (c.lane() == Ctx::WS - 1) sh.bcast[6] = incl;
            }
            c.sync();
            const int n_surv = sh.bcast[6];
            unsigned long long* dst = n_surv <= SURV_CAP ? sh.surv : ws.surv_g;     // the rare big sets (heap still filling) go through global memory
            for (int r = 0; r < rounds; r++) {
                int j = r * NT + c.tid(); int sl = r * NW + c.warp(); unsigned bm = sh.ballots[0][sl];
                if ((bm >> c.lane()) & 1u) dst[sh.bprefix[sl] + popc(bm & c.lanemask_lt())] = kv_pack(sh.cand_s[j], sh.score[j]);
            }
            pend = n_surv;
        }
        c.sync();
    }
    if (c.tid() == 0 && pend) drain();
    c.sync();
    const int n = sh.heap_size;
    for (int i = c.tid(); i < n; i += NT) { out_doc[i] = sh.IFX_HD(i); out_score[i] = sh.IFX_HP(i); }
    if (c.tid() == 0) out_n[0] = n;
    c.sync();
}

// ---------------------------------------------------------------------------------------------------------------
// s1_finish: PopulateResultHeapFromPruning + TopKHeap.GetTopK + ConsolidateSegments: order by (score desc, key asc).
struct FinishShared { float ks[MAX_K]; int32_t kd[MAX_K]; };
IFX_FN void s1_finish(const Ctx& c, const DevIndex& ix, FinishShared& sh, int64_t* key, int32_t* doc, float* score, int32_t* n_io) {
    const int NT = c.nthreads(); const int n = n_io[0]; if (n <= 0) return;
    int n2 = 1; while (n2 < n) n2 <<= 1;
    float* ks = sh.ks; int32_t* kd = sh.kd;
    for (int i = c.tid(); i < n2; i += NT) { if (i < n) { ks[i] = score[i]; kd[i] = doc[i]; } else { ks[i] = -1.f; kd[i] = 0x7fffffff; } }
    c.sync();
    auto before = [&](int a, int b) -> bool {   // a ranks before b
        if (ks[a] != ks[b]) return ks[a] > ks[b];
        if (kd[a] == 0x7fffffff || kd[b] == 0x7fffffff) return kd[a] < kd[b];
        return ix.doc_key[kd[a]] < ix.doc_key[kd[b]];
    };
    for (int k = 2; k <= n2; k <<= 1) for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = c.tid(); i < n2; i += NT) { int l = i ^ j; if (l > i) { bool up = (i & k) == 0; bool sw = up ? before(l, i) : before(i, l); if (sw) { float x = ks[i]; ks[i] = ks[l]; ks[l] = x; int y = kd[i]; kd[i] = kd[l]; kd[l] = y; } } }
        c.sync();
    }
    if (ix.key_first) {      // ConsolidateSegments (SegmentProcessor.cs:15-37): the best entry per DocumentKey; the coverage stage then reads the first live document of the key
        if (c.tid() == 0) { int m = 0;
            for (int i = 0; i < n; i++) { const int64_t k = ix.doc_key[kd[i]]; bool seen = false; for (int j = 0; j < m && !seen; j++) seen = ix.doc_key[kd[j]] == k; if (!seen) { kd[m] = kd[i]; ks[m] = ks[i]; m++; } }
            n_io[0] = m; }
        c.sync();
        const int m = n_io[0];
        for (int i = c.tid(); i < m; i += NT) { const int d = ix.key_first[kd[i]]; doc[i] = d; score[i] = ks[i]; key[i] = ix.doc_key[d]; }
        c.sync(); return;
    }
    for (int i = c.tid(); i < n; i += NT) { doc[i] = kd[i]; score[i] = ks[i]; key[i] = ix.doc_key[kd[i]]; }
    c.sync();
}

}  // namespace ifx
