// events_items.cuh — per-receipt device functions of the event path: the events-AMT walk, pass 1's per-receipt decode, the
// receipts-AMT lookup and pass 2's per-match work (reference events/generator.rs:206-301). The kernels that drive them are in
// events.cu; they live in a header so that tests/host_fuzz can run the very same code on the CPU against the oracle.
#pragma once
#include "ipld.cuh"
#include "rawcid.cuh"

namespace ipcfp {

// ------------------------------------------------------------------------------------------ events AMT walk
enum WalkMode { WALK_ANY = 0, WALK_COUNT = 1, WALK_EMIT = 2 };



struct EmitCtx {
    ipcfp_event_proof* proofs;   // base for this match
    uint8_t* blob;               // data blob base (whole result)
    uint64_t blob_off;           // running offset for this match
    uint64_t exec_index;
    RawCid msg_cid;
};
struct WalkOut { uint32_t nproofs; uint32_t nbytes; bool any; };

__device__ __forceinline__ void emit_proof(const uint8_t* p, const EvLog& ev, uint64_t j, EmitCtx& ec, uint32_t k) {
    ipcfp_event_proof q;
    q.exec_index = ec.exec_index;
    q.event_index = j;
    q.emitter = ev.emitter;
    q.n_topics = ev.ntopics;
    q.data_len = ev.data_len;
    q.topics_off = ec.blob_off;
    uint8_t* o = ec.blob + ec.blob_off;
    for (uint32_t t = 0; t < ev.ntopics; t++) {
        const uint8_t* src = p + topic_offset(ev, t);
        for (int b = 0; b < 32; b++) o[32 * t + b] = src[b];
    }
    ec.blob_off += 32ull * ev.ntopics;
    q.data_off = ec.blob_off;
    o = ec.blob + ec.blob_off;
    for (uint32_t b = 0; b < ev.data_len; b++) o[b] = p[ev.data_off + b];
    ec.blob_off += ev.data_len;
    for (int b = 0; b < 6; b++) q.message_cid[b] = (uint8_t)(ec.msg_cid.w[4] >> (8 * b));
    for (int b = 0; b < 32; b++) q.message_cid[6 + b] = (uint8_t)(ec.msg_cid.w[b >> 3] >> (8 * (b & 7)));
    q._pad[0] = q._pad[1] = 0;
    ec.proofs[k] = q;
}

// Decodes the values of one events-AMT node. Returns false on a decode error (r.err set).
template <int MODE, int WINMODE = 0>
__device__ __forceinline__ void node_events(Rd& r, const uint8_t* p, const AmtNodeHdr& h, uint32_t nv, uint64_t base, const Matcher& m,
                                            WalkOut& wo, EmitCtx* ec, uint32_t tune = 0) {
    for (uint32_t v = 0; v < nv && !r.err; v++) {
        // rolling prefetch: 2 lines ahead of the dependent walk — measured best of 0/2/3/4/6 (profiles/r1_pass1_prefetch_sweep.txt);
        // IPCFP_PASS1_TUNE: bits 4..7 = other distance in lines, bit 1 = off
        const uint32_t ahead = (tune >> 4) & 15u ? 128u * ((tune >> 4) & 15u) : 256u;
        if (!(tune & 2) && r.pos + ahead < r.n) prefetch_l2(r.p + r.pos + ahead);
        if ((tune & 1) && r.pos + 128 < r.n) prefetch_l1(r.p + r.pos + 128);  // experiment: next line into L1
        EvLog ev;
        decode_stamped_event<WINMODE>(r, ev);
        if (r.err) break;
        if (event_matches(p, ev, m)) {
            wo.any = true;
            if (MODE != WALK_ANY) {
                uint64_t j = base + bm_select(h.bm, v);
                if (MODE == WALK_EMIT) emit_proof(p, ev, j, *ec, wo.nproofs);
                wo.nproofs++;
                wo.nbytes += 32 * ev.ntopics + ev.data_len;
            }
        }
    }
}

// Full in-order walk of Amt<StampedEvent> (v3) rooted at block root_blk — `for_each` of
// fvm_ipld_amt [UPSTREAM]: every reachable node is loaded through the store (and recorded when
// wbits != nullptr). Returns 0 ok, else DevCode; detail in *detail.
template <int MODE>
static __device__ __noinline__ uint32_t walk_events(const StoreView* sp, uint32_t root_blk, const Matcher* mp, uint32_t* wbits, WalkOut& wo, EmitCtx* ec,
                                uint32_t* detail) {
    const StoreView& s = *sp;
    const Matcher m = *mp;
    struct Frame { uint32_t blk; uint32_t k; uint64_t base; };
    Frame stk[66];
    int depth = 0;
    stk[0].blk = root_blk; stk[0].k = 0; stk[0].base = 0;
    uint32_t bw = 3, height = 0;
    while (depth >= 0) {
        Frame& f = stk[depth];
        uint32_t len;
        const uint8_t* p = store_block(s, f.blk, len);
        Rd r(p, len);
        if (depth == 0) { uint64_t cnt; amt_root_begin(r, 3, bw, height, cnt); }
        uint32_t lvl = height - (uint32_t)depth;
        AmtNodeHdr h;
        amt_node_begin(r, bw, h);
        if (f.k == 0) {
            uint32_t nv = rd_array(r);
            node_events<MODE>(r, p, h, nv, f.base, m, wo, ec);
            amt_node_finish(r, h, nv, lvl);
            if (r.err) { *detail = r.err; return DC_DECODE; }
        } else if (r.err) { *detail = r.err; return DC_DECODE; }
        if (h.nl == 0 || f.k >= h.nl) { depth--; continue; }
        uint32_t slot = bm_select(h.bm, f.k);
        int32_t child = store_lookup(s, p + h.links_off + 43 * f.k + 5);
        if (child < 0) { *detail = 0; return DC_MISSING; }
        if (wbits) witness_mark(s, wbits, (uint32_t)child);
        uint64_t cbase = f.base + (uint64_t)slot * pow_sat(bw, lvl);
        f.k++;
        depth++;
        stk[depth].blk = (uint32_t)child; stk[depth].k = 0; stk[depth].base = cbase;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------ pass 1
struct Pass1Args {
    StoreView store;
    const StoreView* store_dev;    // same view in device memory (for the out-of-line walker)
    const Matcher* m_dev;
    Matcher m;
    const uint8_t* events_roots;
    const uint8_t* has_root;
    uint64_t lo, hi;
    uint32_t* match_bits;          // bit (i - lo)
    uint32_t* cnt;                 // [i - lo] matching events of receipt i  (EventProof count of pass 2)
    uint32_t* nbytes;              // [i - lo] topics+data bytes of those events
    unsigned long long* err;
    unsigned long long* stats;     // [0] nodes scanned, [1] bytes scanned
    uint32_t tune;                 // experiment bits (env IPCFP_PASS1_TUNE), 0 = default
};

// ------------------------------------------------------------------------------------------ receipts AMT
// Amtv0<Receipt>::get(i) with recording (events/generator.rs:249). 1 = Some, 0 = None, <0 = -DevCode.
static __device__ int receipts_get(const StoreView& s, uint32_t root_blk, uint64_t i, uint32_t* wbits, uint32_t* detail) {
    uint32_t len;
    const uint8_t* p = store_block(s, root_blk, len);
    Rd r(p, len);
    uint32_t bw, height;
    uint64_t cnt;
    amt_root_begin(r, 0, bw, height, cnt);
    if (r.err) { *detail = r.err; return -(int)DC_DECODE; }
    if (i >= pow_sat(3, height + 1)) return 0;
    uint32_t lvl = height;
    for (;;) {
        AmtNodeHdr h;
        amt_node_begin(r, 3, h);
        uint32_t nv = rd_array(r);
        for (uint32_t v = 0; v < nv && !r.err; v++) parse_receipt(r);
        amt_node_finish(r, h, nv, lvl);
        if (r.err) { *detail = r.err; return -(int)DC_DECODE; }
        uint32_t idx = (uint32_t)((i / pow_sat(3, lvl)) & 7);
        if (h.nl == 0) {
            if (lvl != 0) return 0;
            return bm_test(h.bm, idx) ? 1 : 0;
        }
        if (!bm_test(h.bm, idx)) return 0;
        uint32_t k = bm_rank(h.bm, idx);
        int32_t child = store_lookup(s, p + h.links_off + 43 * k + 5);
        if (child < 0) { *detail = 0; return -(int)DC_MISSING; }
        witness_mark(s, wbits, (uint32_t)child);
        p = store_block(s, (uint32_t)child, len);
        r = Rd(p, len);
        lvl--;
    }
}

// ------------------------------------------------------------------------------------------ pass 2
struct Pass2Args {
    StoreView store;
    const StoreView* store_dev;
    const Matcher* m_dev;
    Matcher m;
    const uint8_t* events_roots;
    uint64_t lo;
    const uint32_t* match_rel;     // positions relative to lo, ascending
    uint64_t n_match;
    uint32_t receipts_root_blk;
    const RawCid* exec_cids;       // exec_raw[pos]
    const uint32_t* exec_idx;      // execution order → position in exec_raw
    const unsigned long long* n_exec;
    uint32_t* wbits;
    unsigned long long* err;
    const uint32_t* cnt;           // [i - lo] proofs of receipt i (from pass 1)
    const uint64_t* proof_base;    // [i - lo] exclusive scans over all receipts of the range
    const uint64_t* byte_base;
    ipcfp_event_proof* proofs;
    uint8_t* blob;
    uint32_t* any_skip;            // set when a matching receipt is absent from the receipts AMT
    uint32_t per_warp;             // 1: one matching receipt per warp (lane 0 walks); 0: one per thread
    uint32_t resolve_msg;          // 1: exec.get(i) check + message CID from exec_cids; 0: neither (shard: the execution order spans shards and
                                   // is resolved afterwards — by the caller, or by the in-library protocol with k_check_exec)
};

// One thread per matching receipt (events/generator.rs:242-301): exec.get(i), r_amt.get(i) with path
// recording, full in-order walk of its events AMT with recording, EventProof emission at the
// offsets pass 1 already counted.
__device__ __forceinline__ void pass2_item(const Pass2Args& a, uint64_t t) {
    uint32_t rel = a.match_rel[t];
    uint64_t i = a.lo + rel;
    // exec.get(i) comes first (:244-246)
    if (a.resolve_msg && i >= *a.n_exec) { report_error(a.err, ST_PASS2, i, DC_MISSING_EXEC, 0); return; }
    uint32_t detail = 0;
    int got = receipts_get(a.store, a.receipts_root_blk, i, a.wbits, &detail);
    if (got < 0) { report_error(a.err, ST_PASS2, i, (uint32_t)(-got), detail); return; }
    ipcfp_event_proof* out = a.proofs + a.proof_base[rel];
    if (got == 0) {  // `continue` at :249-251 — the slots pass 1 reserved stay empty and are dropped on the host
        uint32_t c = a.cnt[rel];
        for (uint32_t k = 0; k < c; k++) out[k].exec_index = 0xFFFFFFFFFFFFFFFFull;
        *a.any_skip = 1;
        return;
    }
    int32_t root = store_lookup(a.store, a.events_roots + 38 * i);
    if (root < 0) { report_error(a.err, ST_PASS2, i, DC_MISSING, 0); return; }
    witness_mark(a.store, a.wbits, (uint32_t)root);
    WalkOut wo{0, 0, false};
    EmitCtx ec;
    ec.proofs = out;
    ec.blob = a.blob;
    ec.blob_off = a.byte_base[rel];
    ec.exec_index = i;
    if (a.resolve_msg == 1) ec.msg_cid = a.exec_cids[a.exec_idx[i]]; else ec.msg_cid = RawCid{};
    uint32_t rc = walk_events<WALK_EMIT>(a.store_dev, (uint32_t)root, a.m_dev, a.wbits, wo, &ec, &detail);
    if (rc) report_error(a.err, ST_PASS2, i, rc, detail);
}

// ------------------------------------------------------------------------------------------ several specs in one scan
// ipcfp_generate_event_proof_multi. Every event is decoded once and gives the mask of the specs it matches (event_spec_mask).
// Output layout is spec-major: the (spec, matching receipt) pairs in spec order, receipts ascending within a spec, each pair owning
// a run of proof slots and blob bytes. A pair's index is the rank of bit spec * stride + t (t = position in the list of matching
// receipts) in the pair bitmap.
struct MultiEmit {
    ipcfp_event_proof* proofs;
    uint8_t* blob;
    uint64_t* proof_cur;           // [pair] next proof slot of the pair (starts as the spec-major exclusive scan)
    uint64_t* byte_cur;            // [pair] next blob byte of the pair
    const uint32_t* pair_bits;
    const uint64_t* pair_prefix;   // exclusive popcount prefix of pair_bits' words
    uint64_t stride, t;
    uint64_t exec_index;
    RawCid msg_cid;
};
__device__ __forceinline__ uint64_t pair_index(const uint32_t* bits, const uint64_t* prefix, uint64_t bit) {
    const uint64_t w = bit >> 5;
    return prefix[w] + (uint64_t)__popc(bits[w] & ((1u << (bit & 31)) - 1u));
}

// node_events for a MultiMatcher: `mask` collects the specs that match; counts are summed over specs (an event matching two specs
// is two proofs); WALK_EMIT writes each matching event into the run of every spec it matches
template <int MODE>
__device__ __forceinline__ void node_events_multi(Rd& r, const uint8_t* p, const AmtNodeHdr& h, uint32_t nv, uint64_t base, const MultiMatcher& mm,
                                                  uint64_t& mask, WalkOut& wo, MultiEmit* em) {
    for (uint32_t v = 0; v < nv && !r.err; v++) {
        if (r.pos + 256 < r.n) prefetch_l2(r.p + r.pos + 256);
        EvLog ev;
        decode_stamped_event(r, ev);
        if (r.err) break;
        const uint64_t hit = event_spec_mask(p, ev, mm);
        if (!hit) continue;
        mask |= hit;
        const uint32_t c = (uint32_t)__popcll(hit);
        wo.any = true;
        wo.nproofs += c;
        wo.nbytes += c * (32 * ev.ntopics + ev.data_len);
        if (MODE == WALK_EMIT) {
            const uint64_t j = base + bm_select(h.bm, v);
            for (uint64_t m = hit; m; m &= m - 1) {
                const uint64_t k = (uint64_t)(__ffsll((long long)m) - 1);
                const uint64_t q = pair_index(em->pair_bits, em->pair_prefix, k * em->stride + em->t);
                EmitCtx ec{em->proofs + em->proof_cur[q], em->blob, em->byte_cur[q], em->exec_index, em->msg_cid};
                emit_proof(p, ev, j, ec, 0);
                em->proof_cur[q]++;
                em->byte_cur[q] = ec.blob_off;
            }
        }
    }
}

// walk_events for a MultiMatcher. The matcher (5 KB) stays in memory instead of being copied into registers as walk_events does.
template <int MODE>
static __device__ __noinline__ uint32_t walk_events_multi(const StoreView* sp, uint32_t root_blk, const MultiMatcher* mm, uint32_t* wbits, uint64_t& mask,
                                                          WalkOut& wo, MultiEmit* em, uint32_t* detail) {
    const StoreView& s = *sp;
    struct Frame { uint32_t blk; uint32_t k; uint64_t base; };
    Frame stk[66];
    int depth = 0;
    stk[0].blk = root_blk; stk[0].k = 0; stk[0].base = 0;
    uint32_t bw = 3, height = 0;
    while (depth >= 0) {
        Frame& f = stk[depth];
        uint32_t len;
        const uint8_t* p = store_block(s, f.blk, len);
        Rd r(p, len);
        if (depth == 0) { uint64_t cnt; amt_root_begin(r, 3, bw, height, cnt); }
        uint32_t lvl = height - (uint32_t)depth;
        AmtNodeHdr h;
        amt_node_begin(r, bw, h);
        if (f.k == 0) {
            uint32_t nv = rd_array(r);
            node_events_multi<MODE>(r, p, h, nv, f.base, *mm, mask, wo, em);
            amt_node_finish(r, h, nv, lvl);
            if (r.err) { *detail = r.err; return DC_DECODE; }
        } else if (r.err) { *detail = r.err; return DC_DECODE; }
        if (h.nl == 0 || f.k >= h.nl) { depth--; continue; }
        uint32_t slot = bm_select(h.bm, f.k);
        int32_t child = store_lookup(s, p + h.links_off + 43 * f.k + 5);
        if (child < 0) { *detail = 0; return DC_MISSING; }
        if (wbits) witness_mark(s, wbits, (uint32_t)child);
        uint64_t cbase = f.base + (uint64_t)slot * pow_sat(bw, lvl);
        f.k++;
        depth++;
        stk[depth].blk = (uint32_t)child; stk[depth].k = 0; stk[depth].base = cbase;
    }
    return 0;
}

struct Pass1MultiArgs {
    StoreView store;
    const StoreView* store_dev;
    const MultiMatcher* mm;        // device memory (k_pass1_multi stages a copy in shared memory)
    const uint8_t* events_roots;
    const uint8_t* has_root;
    uint64_t n;                    // receipts
    uint32_t* match_bits;          // bit i: some spec matches receipt i
    uint64_t* spec_mask;           // [i] the specs matching receipt i, written for matching receipts only
    unsigned long long* err;
    unsigned long long* stats;     // [0] nodes scanned, [1] bytes scanned
    unsigned long long* n_proofs;  // Σ over specs of the spec's proofs
    unsigned long long* n_bytes;   // Σ over specs of the spec's topics+data bytes
    unsigned long long* n_pairs;   // Σ over receipts of popcount(spec mask)
};
// pass 1, receipt i, phase 1: Blockstore::get of its events root (pass1_body's)
__device__ __forceinline__ int32_t pass1_multi_lookup(const Pass1MultiArgs& a, uint64_t i) {
    if (i >= a.n || !a.has_root[i]) return -1;
    const int32_t blk = store_lookup(a.store, a.events_roots + 38 * i);
    if (blk < 0) report_error(a.err, ST_PASS1, i, DC_MISSING, 0);
    return blk;
}
// phase 2: decode the events AMT rooted at blk (p, len) once → the receipt's spec mask; proofs and bytes over all specs in wo
__device__ __forceinline__ uint64_t pass1_multi_decode(const Pass1MultiArgs& a, const MultiMatcher& mm, uint64_t i, uint32_t blk, const uint8_t* p,
                                                       uint32_t len, WalkOut& wo) {
    Rd r(p, len);
    uint32_t bw, height;
    uint64_t cnt;
    amt_root_begin(r, 3, bw, height, cnt);
    AmtNodeHdr h;
    amt_node_begin(r, bw, h);
    uint32_t nv = rd_array(r);
    uint64_t mask = 0;
    wo = WalkOut{0, 0, false};
    node_events_multi<WALK_COUNT>(r, p, h, nv, 0, mm, mask, wo, nullptr);
    amt_node_finish(r, h, nv, height);
    if (r.err) { report_error(a.err, ST_PASS1, i, DC_DECODE, r.err); mask = 0; wo = WalkOut{0, 0, false}; }
    else if (h.nl) {
        uint32_t detail = 0;
        mask = 0;
        wo = WalkOut{0, 0, false};
        uint32_t rc = walk_events_multi<WALK_COUNT>(a.store_dev, blk, a.mm, nullptr, mask, wo, nullptr, &detail);
        if (rc) { report_error(a.err, ST_PASS1, i, rc, detail); mask = 0; wo = WalkOut{0, 0, false}; }
    }
    return mask;
}

// proofs and topics+data bytes of pair q: the events AMT of its receipt walked with that spec's matcher alone. Pass 1 has walked
// every one of these AMTs without a fault (or the call has failed already).
__device__ __forceinline__ void pair_count_item(const StoreView& store, const StoreView* store_dev, const MultiMatcher* mm, const uint8_t* events_roots,
                                                const uint32_t* match_rel, const uint32_t* pairs, uint64_t stride, uint64_t q, uint32_t* cnt,
                                                uint32_t* nbytes) {
    const uint64_t pr = pairs[q];
    const uint64_t i = match_rel[pr % stride];
    const int32_t root = store_lookup(store, events_roots + 38 * i);
    WalkOut wo{0, 0, false};
    uint32_t detail = 0;
    if (root >= 0) walk_events<WALK_COUNT>(store_dev, (uint32_t)root, &mm->m[pr / stride], nullptr, wo, nullptr, &detail);
    cnt[q] = wo.nproofs;
    nbytes[q] = wo.nbytes;
}

struct Pass2MultiArgs {
    StoreView store;
    const StoreView* store_dev;
    const MultiMatcher* mm;
    const uint8_t* events_roots;
    const uint32_t* match_rel;     // matching receipts, ascending
    const uint64_t* spec_mask;     // [receipt] from pass 1
    uint64_t n_match;
    uint32_t receipts_root_blk;
    const RawCid* exec_cids;
    const uint32_t* exec_idx;
    const unsigned long long* n_exec;
    uint32_t* wbits;
    unsigned long long* err;
    const uint32_t* pair_bits;
    const uint64_t* pair_prefix;
    uint64_t stride;
    const uint32_t* pair_cnt;      // [pair] proofs of the pair
    uint64_t* proof_cur;           // [pair] spec-major exclusive scans, advanced by pass 2
    uint64_t* byte_cur;
    ipcfp_event_proof* proofs;
    uint8_t* blob;
    uint32_t* any_skip;
    uint32_t per_warp;
};
// pass2_item for every spec of matching receipt t at once: exec.get(i), r_amt.get(i) with recording, ONE recorded walk of the
// events AMT emitting into each spec's run. The reference runs the specs one after another, so a fault at receipt i is met first
// in the call of the lowest spec matching i: the error key carries that spec in bits 32..39 of the index (receipts < 2^32), i.e.
// it is ordered by (spec, i, code, detail).
__device__ __forceinline__ void pass2_multi_item(const Pass2MultiArgs& a, uint64_t t) {
    const uint64_t i = a.match_rel[t];
    const uint64_t mask = a.spec_mask[i];
    const uint64_t ekey = ((uint64_t)(__ffsll((long long)mask) - 1) << 32) | i;
    if (i >= *a.n_exec) { report_error(a.err, ST_PASS2, ekey, DC_MISSING_EXEC, 0); return; }
    uint32_t detail = 0;
    int got = receipts_get(a.store, a.receipts_root_blk, i, a.wbits, &detail);
    if (got < 0) { report_error(a.err, ST_PASS2, ekey, (uint32_t)(-got), detail); return; }
    if (got == 0) {  // `continue` for every spec: the reserved slots stay empty and are dropped on the host
        for (uint64_t m = mask; m; m &= m - 1) {
            const uint64_t q = pair_index(a.pair_bits, a.pair_prefix, (uint64_t)(__ffsll((long long)m) - 1) * a.stride + t);
            for (uint32_t k = 0; k < a.pair_cnt[q]; k++) a.proofs[a.proof_cur[q] + k].exec_index = 0xFFFFFFFFFFFFFFFFull;
        }
        *a.any_skip = 1;
        return;
    }
    int32_t root = store_lookup(a.store, a.events_roots + 38 * i);
    if (root < 0) { report_error(a.err, ST_PASS2, ekey, DC_MISSING, 0); return; }
    witness_mark(a.store, a.wbits, (uint32_t)root);
    MultiEmit em{a.proofs, a.blob, a.proof_cur, a.byte_cur, a.pair_bits, a.pair_prefix, a.stride, t, i, a.exec_cids[a.exec_idx[i]]};
    uint64_t seen = 0;
    WalkOut wo{0, 0, false};
    uint32_t rc = walk_events_multi<WALK_EMIT>(a.store_dev, (uint32_t)root, a.mm, a.wbits, seen, wo, &em, &detail);
    if (rc) report_error(a.err, ST_PASS2, ekey, rc, detail);
}
}  // namespace ipcfp
