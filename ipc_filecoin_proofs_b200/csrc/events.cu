// events.cu — the two-pass receipt/event AMT scan on the GPU.
//
// Replaces, for the data-parallel path, reference src/proofs/events/generator.rs:60-307:
//   k_setup            collect_base_witness (:122-145) + TxMeta decode + AMT root loads
//   k_amt_level/...    record_transaction_amts (:148-177) and build_execution_order
//                      (events/utils.rs:33-94) as ONE level-synchronous, order-preserving BFS
//   k_dedup_*          first-seen dedup of the execution order (utils.rs:56-91)
//   k_pass1            find_matching_events pass 1 (:206-239): one thread decodes one events-AMT
//                      root node, tests (actor_id, topic_0, topic_1) on every StampedEvent, the
//                      warp ballots the matching-receipt bitmap
//   k_pass2<EMIT>      pass 2 (:241-301): per matching receipt, receipts-AMT path walk + full
//                      events-AMT walk, witness bits, EventProof records
//   materialize_witness (witness.cu)   WitnessCollector::materialize (:104)
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include <chrono>
#include "engine.cuh"
#include "hashes.cuh"
#include "ipld.cuh"
#include "prims.cuh"
#include "walk.cuh"
#include "events_items.cuh"
#include "pass1_ring.cuh"
#include "pass1_stage.cuh"
#include "rawcid.cuh"

namespace ipcfp {

// ------------------------------------------------------------------------------------------ pass 1 / pass 2 kernels (per-receipt code: events_items.cuh)
// One thread per receipt: resolve its events root CID, decode the root node of its events AMT,
// test every StampedEvent. The common single-node AMT (≤ 2^bw events) never leaves this
// function; taller AMTs fall through to the generic walker.
template <int WINMODE = 0>
__device__ __forceinline__ void pass1_body(const Pass1Args& a) {
    uint64_t i = a.lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool matched = false;
    uint32_t bytes = 0, nodes = 0, np_ = 0, nb_ = 0;
    // phase 1: Blockstore::get of the events root (hash probe); every lane takes part so the warp
    // can be re-converged before the long decode
    const bool valid = i < a.hi && a.has_root[i];
    int32_t blk = -1;
    if (valid) {
        blk = store_lookup(a.store, a.events_roots + 38 * i);
        if (blk < 0) report_error(a.err, ST_PASS1, i, DC_MISSING, 0);
    }
    uint32_t len = 0;
    const uint8_t* p = nullptr;
    if (blk >= 0) {
        p = store_block(a.store, (uint32_t)blk, len);
        const uint32_t first = (a.tune & 4) ? 2048u : ((a.tune & 8) ? 256u : 512u);
        for (uint32_t o = 0; o < len && o < first; o += 128) prefetch_l2(p + o);  // first lines in flight before the dependent walk
    }
    __syncwarp();
    // phase 2: decode the root node, test every event
    if (blk >= 0) {
        bytes = len + 38; nodes = 1;
        Rd r(p, len);
        uint32_t bw, height;
        uint64_t cnt;
        amt_root_begin(r, 3, bw, height, cnt);
        AmtNodeHdr h;
        amt_node_begin(r, bw, h);
        uint32_t nv = rd_array(r);
        WalkOut wo{0, 0, false};
        node_events<WALK_COUNT, WINMODE>(r, p, h, nv, 0, a.m, wo, nullptr, a.tune);
        amt_node_finish(r, h, nv, height);
        if (r.err) report_error(a.err, ST_PASS1, i, DC_DECODE, r.err);
        else if (h.nl) {
            uint32_t detail = 0;
            wo = WalkOut{0, 0, false};
            uint32_t rc = walk_events<WALK_COUNT>(a.store_dev, (uint32_t)blk, a.m_dev, nullptr, wo, nullptr, &detail);
            if (rc) { report_error(a.err, ST_PASS1, i, rc, detail); wo = WalkOut{0, 0, false}; }
        }
        matched = wo.any;
        np_ = wo.nproofs; nb_ = wo.nbytes;
    }
    if (i < a.hi) { a.cnt[i - a.lo] = np_; a.nbytes[i - a.lo] = nb_; }
    unsigned b = __ballot_sync(0xffffffffu, matched);
    if ((threadIdx.x & 31) == 0) a.match_bits[((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5] = b;
    // per-warp statistics (algorithmic bytes of the scan)
    for (int o = 16; o; o >>= 1) { bytes += __shfl_xor_sync(0xffffffffu, bytes, o); nodes += __shfl_xor_sync(0xffffffffu, nodes, o); }
    if ((threadIdx.x & 31) == 0 && nodes) { atomicAdd(a.stats, (unsigned long long)nodes); atomicAdd(a.stats + 1, (unsigned long long)bytes); }
}
// the same kernel at three register budgets (resident CTAs per SM: 6 → 80 regs, 8 → 64, 10 → 48);
// IPCFP_PASS1_MINB selects one at run time for tuning, 8 is the measured default
__global__ void __launch_bounds__(128, 6) k_pass1(Pass1Args a) { pass1_body(a); }
__global__ void __launch_bounds__(128, 8) k_pass1_occ8(Pass1Args a) { pass1_body(a); }
__global__ void __launch_bounds__(128, 10) k_pass1_occ10(Pass1Args a) { pass1_body(a); }
// windows through two 16-byte loads (2/3 of the L1 wavefronts of three 8-byte loads)
__global__ void __launch_bounds__(128, 8) k_pass1_w16(Pass1Args a) { pass1_body<1>(a); }
__global__ void __launch_bounds__(128, 6) k_pass1_w16_occ6(Pass1Args a) { pass1_body<1>(a); }

// ---- EXPERIMENT (round 2): pass 1 through per-lane shared-memory rings, see pass1_ring.cuh. Same outputs as k_pass1;
// a node the ring path cannot take (malformed head, links = taller AMT) is re-decoded by the arena path below.
template <int CH, int NSLOT>
__global__ void __launch_bounds__(128, (CH * NSLOT <= 256 ? 6 : 3)) k_pass1_ring(Pass1Args a, const uint8_t* arena_end) {
    extern __shared__ __align__(16) uint8_t ring_smem[];
    constexpr uint32_t STRIDE = CH * NSLOT + 16;      // 16-byte aligned rows, 4 banks apart
    uint64_t i = a.lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool matched = false;
    uint32_t bytes = 0, nodes = 0, np_ = 0, nb_ = 0;
    const bool valid = i < a.hi && a.has_root[i];
    int32_t blk = -1;
    if (valid) {
        blk = store_lookup(a.store, a.events_roots + 38 * i);
        if (blk < 0) report_error(a.err, ST_PASS1, i, DC_MISSING, 0);
    }
    uint32_t len = 0;
    const uint8_t* p = nullptr;
    RingWin<CH, NSLOT> ring;
    if (blk >= 0) {
        p = store_block(a.store, (uint32_t)blk, len);
        ring.init(ring_smem + threadIdx.x * STRIDE, p, len, arena_end);
        ring.top_up(0);                                 // first NSLOT chunks in flight before the dependent walk
    }
    __syncwarp();
    if (blk >= 0) {
        bytes = len + 38; nodes = 1;
        WalkOut wo{0, 0, false};
        const bool taken = pass1_ring_item(ring, p, len, a.m, wo);
        if (!taken) {                                    // the arena path decides (and reports) everything about this node
            wo = WalkOut{0, 0, false};
            Rd r(p, len);
            uint32_t bw, height;
            uint64_t cnt;
            amt_root_begin(r, 3, bw, height, cnt);
            AmtNodeHdr h;
            amt_node_begin(r, bw, h);
            uint32_t nv = rd_array(r);
            node_events<WALK_COUNT>(r, p, h, nv, 0, a.m, wo, nullptr, 2u);
            amt_node_finish(r, h, nv, height);
            if (r.err) report_error(a.err, ST_PASS1, i, DC_DECODE, r.err);
            else if (h.nl) {
                uint32_t detail = 0;
                wo = WalkOut{0, 0, false};
                uint32_t rc = walk_events<WALK_COUNT>(a.store_dev, (uint32_t)blk, a.m_dev, nullptr, wo, nullptr, &detail);
                if (rc) { report_error(a.err, ST_PASS1, i, rc, detail); wo = WalkOut{0, 0, false}; }
            }
            if (r.err) wo = WalkOut{0, 0, false};
        }
        matched = wo.any;
        np_ = wo.nproofs; nb_ = wo.nbytes;
    }
    if (i < a.hi) { a.cnt[i - a.lo] = np_; a.nbytes[i - a.lo] = nb_; }
    unsigned b = __ballot_sync(0xffffffffu, matched);
    if ((threadIdx.x & 31) == 0) a.match_bits[((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5] = b;
    for (int o = 16; o; o >>= 1) { bytes += __shfl_xor_sync(0xffffffffu, bytes, o); nodes += __shfl_xor_sync(0xffffffffu, nodes, o); }
    if ((threadIdx.x & 31) == 0 && nodes) { atomicAdd(a.stats, (unsigned long long)nodes); atomicAdd(a.stats + 1, (unsigned long long)bytes); }
}

// exec.get(i) for every matching receipt against the GLOBAL execution order length (sharded calls: the order spans shards)
__global__ void k_check_exec(const uint32_t* __restrict__ match_rel, uint64_t n_match, uint64_t lo, const unsigned long long* __restrict__ n_exec,
                             unsigned long long* err) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_match) return;
    const uint64_t i = lo + match_rel[t];
    if (i >= *n_exec) report_error(err, ST_PASS2, i, 0 /* DC_MISSING_EXEC, ranked before every other code at the same receipt */, 0);
}
// a.per_warp: one matching receipt per WARP (lane 0 walks). A matching receipt is a chain of dependent accesses (hash probe → record →
// strict decode of a 349–413 B node, 7 levels at 1 M receipts, then its events AMT), and 32 lanes on 32 different paths execute that
// chain serialised by divergence: 1 020 matches in 8 CTAs kept 8 of 148 SMs busy for 0.14 ms (profiles/r1_ncu_full_final.txt). One warp
// per match is the shape that took k_read_slots from 0.85 to 0.125 ms (storage.cu); above 16 384 matches the grid fills the machine
// either way and one match per thread is kept. Same per-item code, so results are identical by construction.
__global__ void __launch_bounds__(128) k_pass2(Pass2Args a) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a.per_warp) { if (threadIdx.x & 31) return; t >>= 5; }
    if (t >= a.n_match) return;
    pass2_item(a, t);
}

// ------------------------------------------------------------------------------------------ several specs in one scan (per-item code: events_items.cuh)
// keccak256(event_signature) → m[k].t0 for every spec, one thread per spec (k_setup's thread 96 does it for one)
__global__ void k_spec_keccak(MultiMatcher* mm, const uint8_t* sigs, const uint32_t* sig_off, const uint32_t* sig_len) {
    const uint32_t k = threadIdx.x;
    if (k >= mm->n) return;
    Digest d;
    keccak256(sigs + sig_off[k], sig_len[k], d);
    for (int w = 0; w < 4; w++) mm->m[k].t0[w] = d.w[w];
}
// k_pass1_occ8's thread-per-root shape with every spec tested on every event. The specs are staged in shared memory: the screen of
// event_spec_mask reads two words per spec and event. The ballot gives the bitmap of receipts some spec matches.
__global__ void __launch_bounds__(128, 8) k_pass1_multi(Pass1MultiArgs a) {
    __shared__ MultiMatcher s_mm;
    const uint32_t n_specs = a.mm->n;
    for (uint32_t w = threadIdx.x; w < n_specs * (uint32_t)(sizeof(Matcher) / 8); w += blockDim.x) ((uint64_t*)s_mm.m)[w] = ((const uint64_t*)a.mm->m)[w];
    if (threadIdx.x == 0) s_mm.n = n_specs;
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t blk = pass1_multi_lookup(a, i);
    uint32_t len = 0, bytes = 0, nodes = 0;
    const uint8_t* p = nullptr;
    if (blk >= 0) {
        p = store_block(a.store, (uint32_t)blk, len);
        for (uint32_t o = 0; o < len && o < 512; o += 128) prefetch_l2(p + o);
    }
    __syncwarp();
    uint64_t mask = 0;
    WalkOut wo{0, 0, false};
    if (blk >= 0) {
        bytes = len + 38; nodes = 1;
        mask = pass1_multi_decode(a, s_mm, i, (uint32_t)blk, p, len, wo);
    }
    if (mask) a.spec_mask[i] = mask;
    const unsigned b = __ballot_sync(0xffffffffu, mask != 0);
    if ((threadIdx.x & 31) == 0) a.match_bits[i >> 5] = b;
    uint32_t pairs = (uint32_t)__popcll(mask), np_ = wo.nproofs, nb_ = wo.nbytes;
    for (int o = 16; o; o >>= 1) {
        bytes += __shfl_xor_sync(0xffffffffu, bytes, o); nodes += __shfl_xor_sync(0xffffffffu, nodes, o);
        pairs += __shfl_xor_sync(0xffffffffu, pairs, o); np_ += __shfl_xor_sync(0xffffffffu, np_, o); nb_ += __shfl_xor_sync(0xffffffffu, nb_, o);
    }
    if ((threadIdx.x & 31) == 0 && nodes) { atomicAdd(a.stats, (unsigned long long)nodes); atomicAdd(a.stats + 1, (unsigned long long)bytes); }
    if ((threadIdx.x & 31) == 0 && pairs) {
        atomicAdd(a.n_pairs, (unsigned long long)pairs); atomicAdd(a.n_proofs, (unsigned long long)np_); atomicAdd(a.n_bytes, (unsigned long long)nb_);
    }
}
// bit k * stride + t of the pair bitmap for every spec k matching match t
__global__ void k_pair_bits(const uint32_t* __restrict__ match_rel, const uint64_t* __restrict__ spec_mask, uint64_t n_match, uint64_t stride, uint32_t* pair_bits) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_match) return;
    for (uint64_t m = spec_mask[match_rel[t]]; m; m &= m - 1) {
        const uint64_t bit = (uint64_t)(__ffsll((long long)m) - 1) * stride + t;
        atomicOr(&pair_bits[bit >> 5], 1u << (bit & 31));
    }
}
__global__ void __launch_bounds__(128) k_pair_count(StoreView store, const StoreView* store_dev, const MultiMatcher* mm, const uint8_t* events_roots,
                                                    const uint32_t* match_rel, const uint32_t* pairs, uint64_t n_pairs, uint64_t stride, uint32_t* cnt,
                                                    uint32_t* nbytes) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_pairs) return;
    pair_count_item(store, store_dev, mm, events_roots, match_rel, pairs, stride, q, cnt, nbytes);
}
// per spec k = 0..n_specs: its first pair, proof and blob byte in the spec-major layout (out[k], out[n+1+k], out[2(n+1)+k])
__global__ void k_spec_bounds(const uint32_t* __restrict__ pairs, uint64_t n_pairs, uint64_t stride, const uint64_t* __restrict__ pbase,
                              const uint64_t* __restrict__ bbase, uint64_t n_proofs, uint64_t n_bytes, uint32_t n_specs, uint64_t* out) {
    const uint32_t k = threadIdx.x;
    if (k > n_specs) return;
    uint64_t lo = 0, hi = n_pairs;
    while (lo < hi) { const uint64_t mid = (lo + hi) / 2; if (pairs[mid] < k * stride) lo = mid + 1; else hi = mid; }
    out[k] = lo;
    out[n_specs + 1 + k] = lo < n_pairs ? pbase[lo] : n_proofs;
    out[2 * (n_specs + 1) + k] = lo < n_pairs ? bbase[lo] : n_bytes;
}
// one matching receipt per warp up to 16 384 matches, one per thread above (k_pass2's shapes)
__global__ void __launch_bounds__(128) k_pass2_multi(Pass2MultiArgs a) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a.per_warp) { if (threadIdx.x & 31) return; t >>= 5; }
    if (t >= a.n_match) return;
    pass2_multi_item(a, t);
}

// ------------------------------------------------------------------------------------------ setup + message AMT walk
#define IPCFP_MAX_PARENTS 64
struct SetupArgs {
    StoreView store;
    uint32_t n_parents;
    const uint8_t* parent_cids;    // device copies
    const uint8_t* txmeta_cids;
    const uint8_t* child_cid;      // 38
    const uint8_t* receipts_root;  // 38
    uint32_t skip_tx;
    uint32_t skip_receipts;        // execution-order-only mode: the receipts root is not part of the call
    uint32_t* wbits;
    unsigned long long* err;
    unsigned long long* txerr;     // message-AMT fault word (tx_err_key)
    // outputs
    uint32_t* receipts_root_blk;
    uint32_t* f_blk; uint32_t* f_meta; uint64_t* f_base;  // initial frontier: one item per message AMT
    unsigned long long* f_count;
    uint32_t* amt_height;   // per AMT
    uint64_t* amt_count;    // per AMT (root.count)
    uint32_t* missing_base; // flag: a base-witness CID is not in the store (→ materialize error)
    const uint8_t* sig;     // event signature bytes (zero padded to a multiple of 8) and the Matcher whose t0 this kernel fills
    uint32_t sig_len;
    Matcher* matcher;
};

// One-CTA prologue, the independent pieces on different warps so their dependent lookups overlap:
//   thread 0        Amtv0::<MessageReceipt>::load(&receipts_root) (events/generator.rs:195-196), root validated
//   threads 32..95  one parent each: TxMeta → BLS / SECP AMT roots (seeds the walk frontier, AMT ordinal 2b + k)
//   thread 96       keccak256(event_signature) → Matcher.t0 (EventMatcher::new, events/generator.rs:30-35)
//   threads 128..   base witness marks (parent headers, child header, receipts root, TxMeta blocks)
// Errors go through the atomicMin error word, so the one reported is the one the sequential order meets first.
__global__ void __launch_bounds__(256) k_setup(SetupArgs a) {
    const StoreView& s = a.store;
    const uint32_t t = threadIdx.x, P = a.n_parents;
    if (t >= 128 && !a.skip_tx) {
        for (uint32_t i = t - 128; i < 2 * P + 2; i += 128) {
            const uint8_t* cid = i < P ? a.parent_cids + 38 * i : (i == P ? a.child_cid : (i == P + 1 ? a.receipts_root : a.txmeta_cids + 38 * (i - P - 2)));
            int32_t b = store_lookup(s, cid);
            if (b < 0) *a.missing_base = 1; else witness_mark(s, a.wbits, (uint32_t)b);
        }
    }
    if (t == 96) {
        Digest d;
        keccak256(a.sig, a.sig_len, d);
        a.matcher->t0[0] = d.w[0]; a.matcher->t0[1] = d.w[1]; a.matcher->t0[2] = d.w[2]; a.matcher->t0[3] = d.w[3];
    }
    // TxMeta + message AMT roots (needed for the execution order even when skip_tx). An AMT whose root cannot be loaded keeps
    // a sentinel seed (height / count 0): the walk goes on for the others, and the fault the reference meets FIRST wins the word
    if (t >= 32 && t < 96) for (uint32_t b = t - 32; b < P; b += 64) {
        for (uint32_t k = 0; k < 2; k++) { a.f_meta[2 * b + k] = AMT_SENTINEL; a.f_blk[2 * b + k] = 0; a.f_base[2 * b + k] = 0; a.amt_height[2 * b + k] = 0; a.amt_count[2 * b + k] = 0; }
        int32_t tb = store_lookup(s, a.txmeta_cids + 38 * b);
        if (tb < 0) { report_tx_error(a.txerr, 3 * b, 0, 31, DC_MISSING, 0); continue; }
        if (!a.skip_tx) witness_mark(s, a.wbits, (uint32_t)tb);
        uint32_t len;
        const uint8_t* p = store_block(s, (uint32_t)tb, len);
        Rd r(p, len);
        rd_array_exact(r, 2);
        uint32_t c0 = rd_cid(r), c1 = rd_cid(r);
        rd_end(r);
        if (r.err) { report_tx_error(a.txerr, 3 * b, 0, 31, DC_DECODE, r.err); continue; }
        for (uint32_t k = 0; k < 2; k++) {
            int32_t rb = store_lookup(s, p + (k ? c1 : c0));
            if (rb < 0) { report_tx_error(a.txerr, 3 * b + 1 + k, 0, 31, DC_MISSING, 0); break; }
            if (!a.skip_tx) witness_mark(s, a.wbits, (uint32_t)rb);
            uint32_t rl;
            const uint8_t* rp = store_block(s, (uint32_t)rb, rl);
            Rd rr(rp, rl);
            uint32_t bw, h;
            uint64_t cnt;
            amt_root_begin(rr, 0, bw, h, cnt);
            if (rr.err) { report_tx_error(a.txerr, 3 * b + 1 + k, 0, 31, DC_DECODE, rr.err); break; }
            const uint32_t amt = 2 * b + k;
            a.f_blk[amt] = (uint32_t)rb;
            a.f_meta[amt] = make_meta(amt, 1, h);
            a.f_base[amt] = 0;
            a.amt_height[amt] = h;
            a.amt_count[amt] = cnt;
        }
    }
    if (t != 0) return;
    *a.f_count = 2 * P;
    if (a.skip_receipts) return;
    // Amtv0::<MessageReceipt>::load(&receipts_root, &rec_receipts) (events/generator.rs:195-196)
    int32_t rb = store_lookup(s, a.receipts_root);
    if (rb < 0) { report_error(a.err, ST_RECEIPTS_ROOT, 0, DC_MISSING, 0); return; }
    witness_mark(s, a.wbits, (uint32_t)rb);
    *a.receipts_root_blk = (uint32_t)rb;
    uint32_t len;
    const uint8_t* p = store_block(s, (uint32_t)rb, len);
    Rd r(p, len);
    uint32_t bw, h;
    uint64_t cnt;
    amt_root_begin(r, 0, bw, h, cnt);
    AmtNodeHdr hd;
    amt_node_begin(r, 3, hd);
    uint32_t nv = rd_array(r);
    for (uint32_t v = 0; v < nv && !r.err; v++) parse_receipt(r);
    amt_node_finish(r, hd, nv, h);
    if (r.err) report_error(a.err, ST_RECEIPTS_ROOT, 0, DC_DECODE, r.err);
}

// ---- message-AMT walk, general form: kernels (per-item code: walk.cuh) --------------------------------------
__global__ void __launch_bounds__(128) k_amt_count(StoreView store, Frontier in, const unsigned long long* in_count, uint32_t round, uint32_t last_round,
                                                   uint32_t cap, uint32_t* counts, const uint64_t* rlo, const uint64_t* rhi) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t cnt = *in_count;
    if (cnt > cap) cnt = cap;
    if (t >= cnt) { counts[t] = 0; return; }   // the grid covers exactly the scanned range
    counts[t] = amt_item_count(store, in.blk[t], in.meta[t], in.base[t], round, last_round, rlo, rhi);
}
__global__ void __launch_bounds__(128) k_amt_expand(ExpandArgs a, const uint32_t* counts, unsigned long long* out_count, const unsigned long long* total) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t t = g >> 3;          // frontier item
    const uint32_t j = (uint32_t)g & 7; // lane of the item
    uint64_t cnt = *a.in_count;
    if (cnt > a.cap) cnt = a.cap;
    if (g == 0) {
        unsigned long long n = *total;
        if (a.round < a.last_round && n > a.cap) { report_tx_error(a.err, IPCFP_TX_EIDX_NONE, 0, 0, DC_UNSUPPORTED, 1); n = a.cap; }
        *out_count = n;
    }
    if (t >= cnt) return;
    amt_item_expand(a, t, j, a.in.blk[t], a.in.meta[t], a.in.base[t], counts[t]);
}

// Rounds whose frontier is guaranteed to fit one CTA (≤ 1024 items) run fused in a single launch:
// count, block-wide scan and expand per level with __syncthreads between levels.
#define TOP_CAP 1024
__global__ void __launch_bounds__(TOP_CAP) k_amt_top(ExpandArgs a0, Frontier ping, Frontier pong, unsigned long long* count_io, uint32_t first_round,
                                                      uint32_t n_rounds, uint64_t* scan_tmp) {
    __shared__ uint32_t s_cnt[TOP_CAP];
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_total;
    const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
    Frontier cur = ping, nxt = pong;
    for (uint32_t rr = 0; rr < n_rounds; rr++) {
        uint32_t round = first_round + rr;
        uint64_t cnt = *count_io;
        if (cnt > TOP_CAP) cnt = TOP_CAP;
        uint32_t c = t < cnt ? amt_item_count(a0.store, cur.blk[t], cur.meta[t], cur.base[t], round, a0.last_round, a0.rlo, a0.rhi) : 0;
        // block exclusive scan of c
        uint32_t x = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (uint32_t)o) x += y; }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t v = s_warp[lane], w = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= (uint32_t)o) w += y; }
            s_warp[lane] = w - v;
            if (lane == 31) s_total = w;
        }
        __syncthreads();
        uint32_t ex = s_warp[warp] + x - c;
        scan_tmp[t] = ex;
        s_cnt[t] = c;
        __syncthreads();
        ExpandArgs a = a0;
        a.in = cur; a.out = nxt; a.round = round; a.out_off = scan_tmp;
        for (uint32_t it = t >> 3; it < cnt; it += TOP_CAP / 8) amt_item_expand(a, it, t & 7, cur.blk[it], cur.meta[it], cur.base[it], s_cnt[it]);
        __syncthreads();
        if (t == 0) {
            unsigned long long n = s_total;
            if (round < a0.last_round && n > a0.cap) { report_tx_error(a0.err, IPCFP_TX_EIDX_NONE, 0, 0, DC_UNSUPPORTED, 1); n = a0.cap; }
            *count_io = n;
        }
        __threadfence();
        __syncthreads();
        Frontier tmp = cur; cur = nxt; nxt = tmp;
    }
}

// n_rounds == 1: any grid. n_rounds > 1: ONE CTA walks several small levels back to back (barrier between levels).
__global__ void __launch_bounds__(1024) k_amt_dense(DenseArgs a, uint32_t first_round, uint32_t n_rounds) {
    for (uint32_t rr = 0; rr < n_rounds; rr++) {
        const uint32_t round = first_round + rr;
        if (*(volatile uint32_t*)a.fail) return;        // same value in every thread: written before the previous barrier / launch
        const Frontier in = (round & 1) ? a.pong : a.ping, out = (round & 1) ? a.ping : a.pong;
        const uint64_t n8 = (uint64_t)a.ftot[round] * 8;
        for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n8; g += (uint64_t)gridDim.x * blockDim.x)
            amt_item_dense(a, in, out, round, (uint32_t)(g >> 3), (uint32_t)g & 7);
        if (n_rounds > 1) { __threadfence(); __syncthreads(); }
    }
}

// first-seen dedup of the raw execution list (events/utils.rs:56-91): hash set keyed by the full
// CID holding the smallest position; an entry survives iff it holds its own position.
__global__ void k_dedup_insert(const RawCid* __restrict__ raw, uint64_t n, unsigned long long* table, uint64_t mask) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RawCid c = raw[i];
    uint64_t h = rawcid_hash(c);
    uint32_t fp = (uint32_t)(h >> 32) | 1u;
    unsigned long long mine = ((unsigned long long)fp << 32) | (unsigned long long)(i + 1);
    uint64_t slot = h & mask;
    for (;;) {
        unsigned long long e = table[slot];
        if (e == 0) { e = atomicCAS(&table[slot], 0ull, mine); if (e == 0) return; }
        if ((uint32_t)(e >> 32) == fp && rawcid_eq(raw[(uint32_t)e - 1], c)) { atomicMin(&table[slot], mine); return; }
        slot = (slot + 1) & mask;
    }
}
__global__ void k_dedup_flags(const RawCid* __restrict__ raw, uint64_t n, const unsigned long long* __restrict__ table, uint64_t mask,
                              uint32_t* keep_bits) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool keep = false;
    if (i < n) {
        RawCid c = raw[i];
        uint64_t h = rawcid_hash(c);
        uint32_t fp = (uint32_t)(h >> 32) | 1u;
        uint64_t slot = h & mask;
        for (;;) {
            unsigned long long e = table[slot];
            if (e == 0) break;  // cannot happen: every entry was inserted
            if ((uint32_t)(e >> 32) == fp && rawcid_eq(raw[(uint32_t)e - 1], c)) { keep = ((uint32_t)e - 1) == (uint32_t)i; break; }
            slot = (slot + 1) & mask;
        }
    }
    __syncwarp();
    unsigned b = __ballot_sync(0xffffffffu, keep);
    if ((threadIdx.x & 31) == 0) keep_bits[i >> 5] = b;
}

// ------------------------------------------------------------------------------------------ host orchestration
struct EventResultBox {
    ipcfp_event_result r;  // must stay first
    PinnedArray matching, proofs, blob;
    WitnessOut wit;
    PinnedArray union_host;       // sharded calls with IPCFP_SHARDED_UNION_TO_HOST
    AsyncBuf<RawCid> shard_exec;  // shard mode: this shard's slice of the raw execution list, kept on the device
};

static void throw_device_error(uint64_t key) {
    uint32_t stage = (uint32_t)(key >> 56), code = (uint32_t)(key >> 8) & 0xff, detail = (uint32_t)key & 0xff;
    uint64_t index = (key >> 16) & 0xFFFFFFFFFFull;
    ipcfp_status st;
    const char* what;
    switch (code) {
        case DC_MISSING: st = IPCFP_ERR_MISSING_BLOCK; what = "missing block"; break;
        case DC_DECODE: st = IPCFP_ERR_DECODE; what = "decode error"; break;
        case 0:
        case DC_MISSING_EXEC: st = IPCFP_ERR_MISSING_EXEC; what = "Missing message at index"; break;
        case DC_UNSUPPORTED: st = IPCFP_ERR_UNSUPPORTED; what = "unsupported input (frontier overflow)"; break;
        default: st = IPCFP_ERR_DECODE; what = "error"; break;
    }
    uint64_t out_index = UINT64_MAX;
    const char* stage_name = "?";
    switch (stage) {
        case ST_TXMETA:
            stage_name = "message AMTs";
            if (index != 0xFFFFFFFFFFull && index % 3 == 0 && code == DC_MISSING) out_index = index / 3;  // missing TxMeta of parent b
            break;
        case ST_RECEIPTS_ROOT: stage_name = "receipts AMT root"; break;
        case ST_PASS1: stage_name = "pass 1"; out_index = index; break;
        case ST_PASS2: stage_name = "pass 2"; out_index = index; break;
        case ST_WITNESS: stage_name = "materialize"; break;
        default: break;
    }
    throw Error(st, std::string(what) + " in " + stage_name + " (detail " + std::to_string(detail) + ")", out_index);
}

// message-AMT fault word (tx_err_key, common.cuh)
static void throw_tx_error(uint64_t key) {
    const uint32_t eidx = (uint32_t)(key >> 56), code = (uint32_t)(key >> 4) & 7, detail = (uint32_t)key & 15;
    ipcfp_status st;
    const char* what;
    switch (code) {
        case DC_MISSING: st = IPCFP_ERR_MISSING_BLOCK; what = "missing block"; break;
        case DC_UNSUPPORTED: st = IPCFP_ERR_UNSUPPORTED; what = "unsupported input (frontier overflow)"; break;
        default: st = IPCFP_ERR_DECODE; what = "decode error"; break;
    }
    uint64_t out_index = UINT64_MAX;
    if (eidx != IPCFP_TX_EIDX_NONE && eidx % 3 == 0 && code == DC_MISSING) out_index = eidx / 3;   // missing TxMeta of parent b
    throw Error(st, std::string(what) + " in message AMTs (detail " + std::to_string(detail) + ")", out_index);
}
// the failure the reference's sequential order meets first: message-AMT stage before everything else
static void check_device_errors(const uint64_t* hw) {
    if (hw[15] != IPCFP_NO_ERROR) throw_tx_error(hw[15]);
    if (hw[0] != IPCFP_NO_ERROR) throw_device_error(hw[0]);
}

void tipset_upload(Store* s, const ipcfp_tipset_desc* t, TipsetDev& td) {
    s->use();
    if (!t || !t->child_cid || !t->receipts_root || (t->n_parents && (!t->parent_cids || !t->parent_txmeta_cids)))
        throw Error(IPCFP_ERR_INVALID_ARG, "tipset descriptor has null fields");
    if (t->n_parents > IPCFP_MAX_PARENTS) throw Error(IPCFP_ERR_UNSUPPORTED, "too many parent blocks");
    if (t->n_receipts >= 0xffffffffull) throw Error(IPCFP_ERR_UNSUPPORTED, "more than 2^32 receipts");
    if (t->n_receipts && (!t->events_roots || !t->has_events_root)) throw Error(IPCFP_ERR_INVALID_ARG, "events roots missing");
    td.parent_epoch = t->parent_epoch; td.child_epoch = t->child_epoch; td.n_parents = t->n_parents;
    td.parent_cids.assign(t->parent_cids, t->parent_cids + 38ull * t->n_parents);
    td.txmeta_cids.assign(t->parent_txmeta_cids, t->parent_txmeta_cids + 38ull * t->n_parents);
    memcpy(td.child_cid, t->child_cid, 38);
    memcpy(td.receipts_root, t->receipts_root, 38);
    td.has_state_root = t->child_parent_state_root != nullptr;
    if (td.has_state_root) memcpy(td.child_state_root, t->child_parent_state_root, 38);
    td.n_receipts = t->n_receipts;
    td.events_roots.alloc(t->n_receipts * 38 + 64);
    td.has_root.alloc(t->n_receipts + 64);
    if (t->n_receipts) {
        IPCFP_CUDA(cudaMemcpyAsync(td.events_roots.p, t->events_roots, t->n_receipts * 38, cudaMemcpyHostToDevice, s->stream));
        IPCFP_CUDA(cudaMemcpyAsync(td.has_root.p, t->has_events_root, t->n_receipts, cudaMemcpyHostToDevice, s->stream));
    }
}

ipcfp_event_result* generate_event_proof(Store* s, const ipcfp_tipset_desc* /*t*/, TipsetDev& td, const ipcfp_event_spec* spec, uint32_t flags,
                                         bool sharded, uint64_t lo, uint64_t hi, uint32_t world, uint32_t rank, Comm* comm, ExecOrderOut* exo,
                                         const MultiSpecs* ms) {
    s->use();
    cudaStream_t st = s->stream;
    const auto t_enter = std::chrono::steady_clock::now();
    static thread_local std::chrono::steady_clock::time_point t_last_exit = t_enter;
    // ms: several specs in one scan (ipcfp_generate_event_proof_multi). Setup, walk, dedup and witness are the single call's; the
    // matcher staging, pass 1, the (spec, match) counts and scans, pass 2 and the error order are its own.
    const uint32_t K = ms ? ms->n : 1;
    if (ms) {
        if (!ms->specs || !ms->match_off || !ms->proof_off) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        if (K == 0 || K > IPCFP_MAX_EVENT_SPECS) throw Error(IPCFP_ERR_INVALID_ARG, "n_specs must be 1..IPCFP_MAX_EVENT_SPECS");
        if (sharded || comm || exo || (flags & (IPCFP_SHARDED_UNION_TO_HOST | IPCFP_SHARDED_UNION_FULL)))
            throw Error(IPCFP_ERR_INVALID_ARG, "the multi-spec call is not sharded");
        for (uint32_t k = 0; k < K; k++)
            if (!ms->specs[k].event_signature || !ms->specs[k].topic_1) throw Error(IPCFP_ERR_INVALID_ARG, "event spec has null fields");
        spec = &ms->specs[0];
    }
    if (!spec || !spec->event_signature || !spec->topic_1) throw Error(IPCFP_ERR_INVALID_ARG, "event spec has null fields");
    if (!sharded) { lo = 0; hi = td.n_receipts; }
    if (lo > hi || hi > td.n_receipts) throw Error(IPCFP_ERR_INVALID_ARG, "receipt range out of bounds");
    const uint64_t N = hi - lo;
    const uint64_t nblk = s->n;
    const bool skip_tx = (flags & IPCFP_SCAN_SKIP_TX_AMTS) != 0;
    // comm != nullptr: this call is one shard of a multi-GPU call and runs the cross-shard protocol itself (parallel.cu). Failures
    // are then not thrown where they are seen: every rank keeps taking part in the collectives and all ranks fail together, with
    // the error the reference's sequential order meets first across ALL shards.
    std::unique_ptr<ShardExchange> xch;
    if (comm) {
        if (!sharded) throw Error(IPCFP_ERR_INVALID_ARG, "communicator given for an unsharded call");
        if (s->class_prefix.size() > 1) throw Error(IPCFP_ERR_UNSUPPORTED, "sharded calls need a store with one CID prefix");
        xch.reset(new ShardExchange(comm, s, lo, hi));
    }
    uint64_t pend_tx = IPCFP_NO_ERROR, pend_err = IPCFP_NO_ERROR;   // first failure seen so far (xch mode)
    auto note_errors = [&](const uint64_t* hwp) {
        if (!xch) { check_device_errors(hwp); return; }
        pend_tx = std::min<uint64_t>(pend_tx, hwp[15]);
        pend_err = std::min<uint64_t>(pend_err, hwp[0]);
    };
    auto throw_global = [&](uint64_t gtx, uint64_t gerr, bool gmissing) {
        if (gtx != IPCFP_NO_ERROR) throw_tx_error(gtx);
        if (gerr != IPCFP_NO_ERROR) throw_device_error(gerr);
        if (gmissing) throw Error(IPCFP_ERR_MISSING_BLOCK, "missing block (base witness CID not in the store)");
    };
    unsigned long long* dw = s->dev_words.p;  // [0] err, [1..] counters
    uint64_t* hw = s->host_words.p;

    IPCFP_CUDA(cudaEventRecord(s->ev[0], st));
    IPCFP_CUDA(cudaMemsetAsync(dw, 0xff, 8, st));
    IPCFP_CUDA(cudaMemsetAsync(dw + 1, 0, 40 * 8, st));
    IPCFP_CUDA(cudaMemsetAsync(dw + 15, 0xff, 8, st));   // message-AMT fault word

    // ---- matcher(s)
    auto make_matcher = [](const ipcfp_event_spec* sp) {
        Matcher m;
        memset(&m, 0, sizeof m);
        size_t n1 = strlen(sp->topic_1);
        uint8_t t1[32];
        memset(t1, 0, 32);
        memcpy(t1, sp->topic_1, n1 < 32 ? n1 : 32);  // ascii_to_bytes32 (evm.rs:72-78)
        memcpy(m.t1, t1, 32);
        m.actor = sp->actor_id_filter;
        m.has_actor = sp->has_actor_id_filter ? 1 : 0;
        return m;
    };
    Matcher mh = make_matcher(spec);
    // spec + tipset CIDs go up in ONE copy from the store's pinned staging block (no host sync):
    //   [0,1024) Matcher (t0 is filled in on the device) | signature, zero padded | parent, TxMeta, child, receipts-root CIDs
    // several specs: [0, head) MultiMatcher + the signatures' offsets and lengths | the K signatures, each zero padded | CIDs
    const size_t MULTI_SIGS = (sizeof(MultiMatcher) + 7) & ~(size_t)7;
    const size_t head = ms ? (MULTI_SIGS + 2 * 4 * IPCFP_MAX_EVENT_SPECS + 63) & ~(size_t)63 : 1024;
    std::vector<size_t> sig_at(K + 1, 0);
    for (uint32_t k = 0; k < K; k++) sig_at[k + 1] = sig_at[k] + ((strlen(ms ? ms->specs[k].event_signature : spec->event_signature) + 64) & ~(size_t)63);
    const size_t siglen = strlen(spec->event_signature);
    const size_t sig_cap = sig_at[K];
    const size_t cids_bytes = 38ull * (2 * td.n_parents + 2);
    const size_t small_bytes = head + sig_cap + cids_bytes + 64;
    static_assert(sizeof(Matcher) <= 1024, "Matcher must fit its staging slot");
    const size_t STAGE_TABLES = 32768;                    // second half of the staging block: dense-walk tables
    const size_t tables_off = std::max<size_t>(STAGE_TABLES, (small_bytes + 63) & ~(size_t)63);
    if (!s->stage.p || s->stage.cap < tables_off + STAGE_TABLES) s->stage = PinnedArray(s->pool, tables_off + STAGE_TABLES);
    AsyncBuf<uint8_t> small(small_bytes, st);
    uint8_t* d_sig = small.p + head;                       // 8-byte aligned
    uint8_t* d_cids = small.p + head + sig_cap;
    Matcher* d_matcher = (Matcher*)small.p;
    MultiMatcher* d_mm = (MultiMatcher*)small.p;
    {
        uint8_t* hs = s->stage.as<uint8_t>();
        memset(hs, 0, small_bytes);
        if (ms) {
            MultiMatcher* mm = (MultiMatcher*)hs;
            uint32_t* so = (uint32_t*)(hs + MULTI_SIGS);
            mm->n = K;
            for (uint32_t k = 0; k < K; k++) {
                mm->m[k] = make_matcher(&ms->specs[k]);
                so[k] = (uint32_t)sig_at[k];
                so[IPCFP_MAX_EVENT_SPECS + k] = (uint32_t)strlen(ms->specs[k].event_signature);
                memcpy(hs + head + sig_at[k], ms->specs[k].event_signature, so[IPCFP_MAX_EVENT_SPECS + k]);
            }
        } else {
            memcpy(hs, &mh, sizeof(Matcher));
            memcpy(hs + head, spec->event_signature, siglen);
        }
        uint8_t* hc = hs + head + sig_cap;
        memcpy(hc, td.parent_cids.data(), td.parent_cids.size()); hc += td.parent_cids.size();
        memcpy(hc, td.txmeta_cids.data(), td.txmeta_cids.size()); hc += td.txmeta_cids.size();
        memcpy(hc, td.child_cid, 38); hc += 38;
        memcpy(hc, td.receipts_root, 38);
        IPCFP_CUDA(cudaMemcpyAsync(small.p, hs, small_bytes, cudaMemcpyHostToDevice, st));
    }

    // ---- witness bitmap + setup
    AsyncBuf<uint32_t> wbits((nblk + 31) / 32 + 8, st);
    wbits.zero();
    const uint32_t namt_max = 2 * td.n_parents;
    const uint64_t cap = 4 * nblk + 1024;
    AsyncBuf<uint32_t> fA_blk(cap, st), fA_meta(cap, st), fB_blk(cap, st), fB_meta(cap, st);
    AsyncBuf<uint64_t> fA_base(cap, st), fB_base(cap, st);
    AsyncBuf<uint32_t> misc(64 + 2 * IPCFP_MAX_PARENTS, st);
    AsyncBuf<uint64_t> amt_count(2 * IPCFP_MAX_PARENTS, st);
    misc.zero();
    SetupArgs sa;
    sa.store = s->view; sa.n_parents = td.n_parents;
    sa.parent_cids = d_cids; sa.txmeta_cids = d_cids + 38ull * td.n_parents;
    sa.child_cid = d_cids + 76ull * td.n_parents; sa.receipts_root = sa.child_cid + 38;
    sa.skip_tx = skip_tx; sa.skip_receipts = exo ? 1 : 0; sa.wbits = wbits.p; sa.err = dw; sa.txerr = dw + 15;
    sa.receipts_root_blk = misc.p; sa.missing_base = misc.p + 1; sa.amt_height = misc.p + 64;
    sa.f_blk = fA_blk.p; sa.f_meta = fA_meta.p; sa.f_base = fA_base.p; sa.f_count = dw + 1;
    sa.amt_count = amt_count.p;
    sa.sig = d_sig; sa.sig_len = (uint32_t)siglen; sa.matcher = d_matcher;
    k_setup<<<1, 256, 0, st>>>(sa); IPCFP_LAUNCH_CHECK();
    if (ms) {
        const uint32_t* so = (const uint32_t*)(small.p + MULTI_SIGS);
        k_spec_keccak<<<1, IPCFP_MAX_EVENT_SPECS, 0, st>>>(d_mm, d_sig, so, so + IPCFP_MAX_EVENT_SPECS); IPCFP_LAUNCH_CHECK();
    }
    IPCFP_CUDA(cudaMemcpyAsync(hw + 400, d_matcher, 32, cudaMemcpyDeviceToHost, st));   // t0 → hw[400..404)
    IPCFP_CUDA(cudaMemcpyAsync(hw + 24, misc.p, (64 + 2 * IPCFP_MAX_PARENTS) * 4, cudaMemcpyDeviceToHost, st));
    IPCFP_CUDA(cudaMemcpyAsync(hw + 128, amt_count.p, 2 * IPCFP_MAX_PARENTS * 8, cudaMemcpyDeviceToHost, st));
    IPCFP_CUDA(cudaMemcpyAsync(hw, dw, 16 * 8, cudaMemcpyDeviceToHost, st));
    IPCFP_CUDA(cudaStreamSynchronize(st));
    // A fault seen by the prologue (TxMeta / AMT root / receipts root) is NOT thrown yet: the reference walks the message AMTs
    // before it loads the receipts root, and a fault inside an earlier AMT precedes a missing later root — walk first (general
    // kernels: they cope with the sentinel seeds), then report the first one in the reference's order.
    const bool early_fault = hw[0] != IPCFP_NO_ERROR || hw[15] != IPCFP_NO_ERROR;
    memcpy(mh.t0, hw + 400, 32);
    const uint32_t* misc_h = (const uint32_t*)(hw + 24);
    const uint32_t receipts_root_blk = misc_h[0];
    const bool missing_base = misc_h[1] != 0;
    uint32_t namt = (uint32_t)hw[1];
    uint32_t last_round = 0;
    for (uint32_t k = 0; k < namt && k < namt_max; k++) last_round = std::max(last_round, misc_h[64 + k]);

    // ---- message AMT BFS (recording + raw execution list)
    IPCFP_CUDA(cudaEventRecord(s->ev[1], st));
    // share of the concatenated ("raw") message list this call walks: everything, or — sharded —
    // [Nraw*lo/N, Nraw*hi/N) expressed as one index range per AMT
    std::vector<uint64_t> h_rng(4 * IPCFP_MAX_PARENTS, 0);
    const uint64_t nraw_total = shard_amt_ranges(namt, (const uint64_t*)(hw + 128), sharded, lo, hi, td.n_receipts, h_rng.data(),
                                                 h_rng.data() + 2 * IPCFP_MAX_PARENTS);
    AsyncBuf<uint32_t> counts(cap + 1024, st);
    AsyncBuf<uint64_t> out_off(cap + 1024, st), scratch(scan_scratch_elems(std::max<uint64_t>(cap, N) + 64) + 64, st);
    unsigned long long *ccount = dw + 1, *ncount = dw + 2, *total_dev = dw + 13;
    const uint32_t frontier_cap = (uint32_t)std::min<uint64_t>(cap, 0xffffffffull);
    AsyncBuf<RawCid> exec_raw;
    uint64_t raw_cap = 0;

    // ---- (a) dense walk: plan the level layout on the host (see k_amt_dense)
    const bool force_general = getenv("IPCFP_BFS_GENERAL") != nullptr;   // read per call: tests toggle it
    DensePlan plan;
    if (namt > 0 && namt <= namt_max && !force_general && !early_fault)
        plan = make_dense_plan(namt, misc_h + 64, (const uint64_t*)(hw + 128), h_rng.data(), h_rng.data() + 2 * IPCFP_MAX_PARENTS, frontier_cap, 8ull * cap,
                               STAGE_TABLES);
    AsyncBuf<uint8_t> d_tables;
    AsyncBuf<uint64_t> d_foff;
    AsyncBuf<uint32_t> d_flen;
    auto run_dense = [&]() {
        // tables: per_amt (u64) | fofs (u32) | ftot (u32) through the pinned staging block
        const size_t nb_amt = plan.per_amt.size() * 8, nb_fofs = plan.fofs.size() * 4, nb_ftot = plan.ftot.size() * 4;
        uint8_t* ht = s->stage.as<uint8_t>() + tables_off;
        memcpy(ht, plan.per_amt.data(), nb_amt);
        memcpy(ht + nb_amt, plan.fofs.data(), nb_fofs);
        memcpy(ht + nb_amt + nb_fofs, plan.ftot.data(), nb_ftot);
        d_tables.alloc(nb_amt + nb_fofs + nb_ftot + 64, st);
        IPCFP_CUDA(cudaMemcpyAsync(d_tables.p, ht, nb_amt + nb_fofs + nb_ftot, cudaMemcpyHostToDevice, st));
        raw_cap = plan.nraw;
        exec_raw.alloc(raw_cap + 64, st);
        exec_raw.zero();   // pool memory is not zeroed: an entry the walk failed to write must never look like a message CID
        DenseArgs da;
        da.store = s->view;
        da.ping = Frontier{fA_blk.p, fA_meta.p, fA_base.p}; da.pong = Frontier{fB_blk.p, fB_meta.p, fB_base.p};
        da.vals = exec_raw.p;
        const uint64_t* pa = (const uint64_t*)d_tables.p;
        da.vbase = pa; da.cnt = pa + namt; da.lo = pa + 2ull * namt; da.hi = pa + 3ull * namt;
        da.fofs = (const uint32_t*)(d_tables.p + nb_amt); da.ftot = (const uint32_t*)(d_tables.p + nb_amt + nb_fofs);
        da.namt = namt; da.record = skip_tx ? 0 : 1; da.wbits = wbits.p; da.fail = (uint32_t*)(dw + 14);
        uint64_t fmax = 1;
        for (uint32_t r = 0; r < plan.rounds; r++) fmax = std::max<uint64_t>(fmax, plan.ftot[r]);
        d_foff.alloc(2 * fmax + 8, st); d_flen.alloc(2 * fmax + 8, st);
        da.f_off[0] = d_foff.p; da.f_off[1] = d_foff.p + fmax; da.f_len[0] = d_flen.p; da.f_len[1] = d_flen.p + fmax;
        uint32_t top = 0;
        while (top < plan.rounds && plan.ftot[top] <= 1024) top++;
        if (top) { k_amt_dense<<<1, 1024, 0, st>>>(da, 0, top); IPCFP_LAUNCH_CHECK(); }
        for (uint32_t r = top; r < plan.rounds; r++) {
            k_amt_dense<<<div_up((uint64_t)plan.ftot[r] * 8, 256), 256, 0, st>>>(da, r, 1); IPCFP_LAUNCH_CHECK();
        }
    };

    // ---- (b) general walk: count → scan → expand per level, any AMT shape, exact errors
    AsyncBuf<uint64_t> d_rng;
    auto run_general = [&]() {
        d_rng.alloc(4 * IPCFP_MAX_PARENTS, st);
        IPCFP_CUDA(cudaMemcpyAsync(d_rng.p, h_rng.data(), h_rng.size() * 8, cudaMemcpyHostToDevice, st));
        IPCFP_CUDA(cudaStreamSynchronize(st));
        Frontier fcur{fA_blk.p, fA_meta.p, fA_base.p}, fnxt{fB_blk.p, fB_meta.p, fB_base.p};
        ccount = dw + 1; ncount = dw + 2;
        ExpandArgs ea;
        ea.store = s->view; ea.last_round = last_round; ea.record = skip_tx ? 0 : 1; ea.wbits = wbits.p; ea.err = dw + 15;
        ea.vals = nullptr; ea.cap = frontier_cap;
        ea.rlo = d_rng.p; ea.rhi = d_rng.p + 2 * IPCFP_MAX_PARENTS;
        // static frontier bound per round: namt * 8^round
        auto bound_of = [&](uint32_t round) { uint64_t b = namt; for (uint32_t k = 0; k < round && b <= cap; k++) b *= 8; return std::min<uint64_t>(b, cap); };
        auto alloc_vals = [&]() {
            raw_cap = std::min<uint64_t>(bound_of(last_round) * 8, 8 * cap);
            exec_raw.alloc(raw_cap + 64, st);
            exec_raw.zero();
            ea.vals = exec_raw.p;
        };
        // fused single-CTA rounds while the static bound fits one CTA
        uint32_t top_rounds = 0;
        while (top_rounds <= last_round && bound_of(top_rounds) <= TOP_CAP) top_rounds++;
        uint32_t round = 0;
        if (top_rounds) {
            if (top_rounds > last_round) alloc_vals();  // the last round is inside the fused kernel
            ExpandArgs a0 = ea;
            a0.in = fcur; a0.in_count = ccount; a0.out = fnxt; a0.round = 0; a0.out_off = out_off.p;
            k_amt_top<<<1, TOP_CAP, 0, st>>>(a0, fcur, fnxt, ccount, 0, top_rounds, out_off.p); IPCFP_LAUNCH_CHECK();
            if (top_rounds & 1) std::swap(fcur, fnxt);
            round = top_rounds;
        }
        for (; round <= last_round; round++) {
            uint64_t items = bound_of(round);
            if (round == last_round) alloc_vals();
            unsigned grid = div_up(std::max<uint64_t>(items, 1), 128);
            k_amt_count<<<grid, 128, 0, st>>>(s->view, fcur, ccount, round, last_round, ea.cap, counts.p, ea.rlo, ea.rhi); IPCFP_LAUNCH_CHECK();
            exclusive_scan_u32(counts.p, out_off.p, (uint64_t)grid * 128, (uint64_t*)total_dev, scratch.p, st);
            ExpandArgs a = ea;
            a.in = fcur; a.in_count = ccount; a.out = fnxt; a.round = round; a.out_off = out_off.p;
            k_amt_expand<<<div_up(std::max<uint64_t>(items, 1) * 8, 128), 128, 0, st>>>(a, counts.p, ncount, total_dev); IPCFP_LAUNCH_CHECK();
            std::swap(fcur, fnxt);
            std::swap(ccount, ncount);
        }
        // *ccount now holds the number of raw execution entries (k_amt_top leaves it in place as well).
    };
    bool dense_used = plan.ok;
    if (dense_used) run_dense(); else run_general();
    IPCFP_CUDA(cudaEventRecord(s->ev[9], st));   // the raw message list of this call is complete (cross-shard exchange waits for it)
    bool xch_early = false;
    if (xch) {
        // EARLY H0: with dense message AMTs the length of this shard's slice is known from the roots alone (plan.nraw), so the peers can
        // agree on the slices while the walk is still running and the whole execution-order exchange goes onto the (high-priority)
        // exchange stream right behind it — it then runs under the witness snapshot, the host's sync and pass 1 instead of after them.
        // A shard that cannot promise its slice yet (sparse AMTs → general walk, a fault in the prologue) says so and EVERY shard takes
        // the late path below; a promise that turns out wrong (the dense walk raised its flag) is repaired after pass 2 (`stale`).
        xch->agree_early(plan.ok && !early_fault, plan.ok ? plan.nraw : 0, nraw_total);
        xch_early = xch->all_early;
        if (xch_early) xch->start_exchange(exec_raw.p, s->ev[9]);
    }
    // Witness snapshot: base witness + every message-AMT block are final at this point — start moving
    // them to the host while pass 1 / pass 2 run (witness.cu).
    WitnessBuilder wbuild(s);
    wbuild.by_ref = (flags & IPCFP_WITNESS_BY_REFERENCE) != 0;
    if (!exo) wbuild.snapshot(wbits.p);
    publish_words(s, 0, 18);   // error word, frontier counters (dw[1]/dw[2]), witness counts (dw[8], dw[9]), dense-walk flag (dw[14]), gather split (dw[16], dw[17])
    IPCFP_CUDA(cudaStreamSynchronize(st));
    if (dense_used && hw[14] != 0) {   // the AMTs are not what the dense walk assumes: redo the walk with the general kernels
        dense_used = false;
        k_setup<<<1, 256, 0, st>>>(sa); IPCFP_LAUNCH_CHECK();   // re-seed the frontier (same outputs as before)
        run_general();
        IPCFP_CUDA(cudaEventRecord(s->ev[9], st));
        if (!exo) wbuild.snapshot(wbits.p);
        publish_words(s, 0, 18);
        IPCFP_CUDA(cudaStreamSynchronize(st));
    }
    const uint32_t ccount_idx = (uint32_t)(ccount - dw);
    note_errors(hw);
    if (!dense_used && hw[ccount_idx] > raw_cap) {
        if (!xch) throw Error(IPCFP_ERR_UNSUPPORTED, "unsupported input (message list longer than the walk's capacity)");
        pend_tx = std::min<uint64_t>(pend_tx, tx_err_key(IPCFP_TX_EIDX_NONE, 0, 0, DC_UNSUPPORTED, 1));
    }
    uint64_t nraw = dense_used ? plan.nraw : std::min<uint64_t>(hw[ccount_idx], raw_cap);
    // early mode: the exchange that is running was fed the PLANNED slice; if the dense walk gave up, the list was rewritten underneath it
    bool xch_stale = xch_early && (!dense_used || nraw != plan.nraw);
    if (xch && !xch_early && (pend_tx != IPCFP_NO_ERROR || pend_err != IPCFP_NO_ERROR)) {
        // this shard has no message list: tell the peers (H0), then fail — with the first error over ALL shards, like them
        xch->agree_slices(pend_tx, pend_err, 0);
        throw_global(xch->g_tx, xch->g_err, false);
    }
    if (!exo) wbuild.start_copy(hw[8], hw[9], hw[16], hw[17]);
    if (xch && !xch_early) {
        // LATE H0 (some shard could not promise its slice before its walk was over): agree on the slices now and start the exchange
        xch->agree_slices(IPCFP_NO_ERROR, IPCFP_NO_ERROR, nraw);
        if (!xch->peers_ok) { IPCFP_CUDA(cudaStreamSynchronize(st)); throw_global(xch->g_tx, xch->g_err, false); }
        xch->start_exchange(exec_raw.p, s->ev[9]);
    }
    AsyncBuf<uint32_t> exec_idx(nraw + 32, st), keep_bits((nraw + 31) / 32 + 8, st);
    unsigned long long* n_exec_dev = dw + 3;
    if (sharded) IPCFP_CUDA(cudaMemsetAsync(n_exec_dev, 0, 8, st));   // execution order is resolved across ranks by the caller
    else if (nraw) {
        uint64_t slots = 64;
        while (slots < 2 * nraw) slots <<= 1;
        AsyncBuf<unsigned long long> dtab(slots, st);
        dtab.zero();
        k_dedup_insert<<<div_up(nraw, 256), 256, 0, st>>>(exec_raw.p, nraw, dtab.p, slots - 1); IPCFP_LAUNCH_CHECK();
        k_dedup_flags<<<div_up((nraw + 31) / 32 * 32, 256), 256, 0, st>>>(exec_raw.p, nraw, dtab.p, slots - 1, keep_bits.p); IPCFP_LAUNCH_CHECK();
        AsyncBuf<uint64_t> wp2((nraw + 31) / 32 + 8, st);
        bitmap_to_indices(keep_bits.p, nraw, exec_idx.p, (uint64_t*)n_exec_dev, wp2.p, scratch.p, st);
    } else IPCFP_CUDA(cudaMemsetAsync(n_exec_dev, 0, 8, st));
    IPCFP_CUDA(cudaEventRecord(s->ev[2], st));
    if (exo) {
        // execution-order-only mode (the batched verifier, verify.cu): hand the order over and stop before the scan
        publish_words(s, 3, 1);
        IPCFP_CUDA(cudaStreamSynchronize(st));
        exo->n_exec = hw[3];
        exo->nraw = nraw;
        exo->exec_raw = std::move(exec_raw);
        exo->exec_idx = std::move(exec_idx);
        return nullptr;
    }

    // ---- PASS 1
    const uint64_t N1 = ms ? 0 : N + 8;   // per-receipt counts: the single-spec pass 1 only
    AsyncBuf<uint32_t> match_bits((N + 31) / 32 + 8, st), cnt(N1, st), nby(N1, st);
    AsyncBuf<uint64_t> pbase(N1, st), bbase(N1, st);
    Pass1Args p1;
    p1.store = s->view; p1.store_dev = s->view_dev.p; p1.m_dev = d_matcher; p1.m = mh; p1.events_roots = td.events_roots.p; p1.has_root = td.has_root.p; p1.lo = lo; p1.hi = hi;
    p1.match_bits = match_bits.p; p1.cnt = cnt.p; p1.nbytes = nby.p; p1.err = dw; p1.stats = dw + 4;
    AsyncBuf<uint64_t> spec_mask(ms ? N + 8 : 0, st);
    if (ms && N) {
        // the measured pass-1 variants (IPCFP_PASS1_*) stay on the single-spec kernel: none of them won
        Pass1MultiArgs pm;
        pm.store = s->view; pm.store_dev = s->view_dev.p; pm.mm = d_mm; pm.events_roots = td.events_roots.p; pm.has_root = td.has_root.p; pm.n = N;
        pm.match_bits = match_bits.p; pm.spec_mask = spec_mask.p; pm.err = dw; pm.stats = dw + 4;
        pm.n_proofs = dw + 7; pm.n_bytes = dw + 12; pm.n_pairs = dw + 20;
        k_pass1_multi<<<div_up(N, 128), 128, 0, st>>>(pm); IPCFP_LAUNCH_CHECK();
    } else if (N) {
        // kernel variant: read per call so that one process can sweep them (tools/profile_step.py)
        //   IPCFP_PASS1_STAGE=<chunk>x<slots>x<chunks per pass>   warp-cooperative shared-memory staging (pass1_stage.cuh)
        //   IPCFP_PASS1_RING=<chunk>x<slots>                      per-lane cp.async rings (pass1_ring.cuh, round-1 experiment)
        //   IPCFP_PASS1_MINB=6|8|10, IPCFP_PASS1_TUNE=<bits>      thread-per-node kernel straight from the arena (round 1)
        const char* stage_env = getenv("IPCFP_PASS1_STAGE");
        const char* ring_env = getenv("IPCFP_PASS1_RING");
        const int minb = getenv("IPCFP_PASS1_MINB") ? atoi(getenv("IPCFP_PASS1_MINB")) : 8;
        p1.tune = (uint32_t)(getenv("IPCFP_PASS1_TUNE") ? atoi(getenv("IPCFP_PASS1_TUNE")) : 0);
        auto launch_stage = [&](auto kern, int warps, size_t warp_bytes) {
            const size_t smem = warps * warp_bytes;
            IPCFP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<div_up(N, 32 * warps), 32 * warps, smem, st>>>(p1);
        };
        auto launch_ring = [&](auto kern, size_t smem) {
            IPCFP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<div_up(N, 128), 128, smem, st>>>(p1, (const uint8_t*)s->arena.p + s->arena.n);
        };
        auto is = [](const char* e, const char* v) { return e && !strcmp(e, v); };
        if (is(stage_env, "lean128x4x1")) launch_stage(k_pass1_stage<128, 4, 1, 4, 3, 1>, 4, StageGeom<128, 4, 1>::WARP_BYTES);
        else if (is(stage_env, "lean128x4x1w2")) launch_stage(k_pass1_stage<128, 4, 1, 2, 6, 1>, 2, StageGeom<128, 4, 1>::WARP_BYTES);
        else if (is(stage_env, "lean64x8x2")) launch_stage(k_pass1_stage<64, 8, 2, 4, 3, 1>, 4, StageGeom<64, 8, 2>::WARP_BYTES);
        else if (is(stage_env, "lean128x4x2")) launch_stage(k_pass1_stage<128, 4, 2, 4, 3, 1>, 4, StageGeom<128, 4, 2>::WARP_BYTES);
        else if (is(stage_env, "128x4x1")) launch_stage(k_pass1_stage<128, 4, 1, 4, 3>, 4, StageGeom<128, 4, 1>::WARP_BYTES);
        else if (is(stage_env, "128x4x1w2")) launch_stage(k_pass1_stage<128, 4, 1, 2, 6>, 2, StageGeom<128, 4, 1>::WARP_BYTES);
        else if (is(stage_env, "128x4x2")) launch_stage(k_pass1_stage<128, 4, 2, 4, 3>, 4, StageGeom<128, 4, 2>::WARP_BYTES);
        else if (is(stage_env, "64x8x2")) launch_stage(k_pass1_stage<64, 8, 2, 4, 3>, 4, StageGeom<64, 8, 2>::WARP_BYTES);
        else if (is(stage_env, "64x4x2")) launch_stage(k_pass1_stage<64, 4, 2, 8, 3>, 8, StageGeom<64, 4, 2>::WARP_BYTES);
        else if (is(stage_env, "256x2x1")) launch_stage(k_pass1_stage<256, 2, 1, 4, 3>, 4, StageGeom<256, 2, 1>::WARP_BYTES);
        else if (is(stage_env, "256x4x1")) launch_stage(k_pass1_stage<256, 4, 1, 2, 3>, 2, StageGeom<256, 4, 1>::WARP_BYTES);
        else if (is(ring_env, "128x2")) launch_ring(k_pass1_ring<128, 2>, 128 * (128 * 2 + 16));
        else if (is(ring_env, "128x4")) launch_ring(k_pass1_ring<128, 4>, 128 * (128 * 4 + 16));
        else if (is(ring_env, "256x2")) launch_ring(k_pass1_ring<256, 2>, 128 * (256 * 2 + 16));
        else if (getenv("IPCFP_PASS1_W16") && atoi(getenv("IPCFP_PASS1_W16")) == 6) k_pass1_w16_occ6<<<div_up(N, 128), 128, 0, st>>>(p1);
        else if (getenv("IPCFP_PASS1_W16")) k_pass1_w16<<<div_up(N, 128), 128, 0, st>>>(p1);
        else if (minb >= 10) k_pass1_occ10<<<div_up(N, 128), 128, 0, st>>>(p1);
        else if (minb >= 8) k_pass1_occ8<<<div_up(N, 128), 128, 0, st>>>(p1);
        else k_pass1<<<div_up(N, 128), 128, 0, st>>>(p1);
        IPCFP_LAUNCH_CHECK();
    }
    IPCFP_CUDA(cudaEventRecord(s->ev[3], st));
    AsyncBuf<uint32_t> match_rel(N + 32, st);
    AsyncBuf<uint64_t> wp3((N + 31) / 32 + 8, st);
    unsigned long long* n_match_dev = dw + 6;
    bitmap_to_indices(match_bits.p, (N + 31) / 32 * 32, match_rel.p, (uint64_t*)n_match_dev, wp3.p, scratch.p, st);
    if (!ms) {
        exclusive_scan_u32(cnt.p, pbase.p, N, (uint64_t*)(dw + 7), scratch.p, st);
        exclusive_scan_u32(nby.p, bbase.p, N, (uint64_t*)(dw + 12), scratch.p, st);
    }
    publish_words(s, 0, ms ? 21 : 16);   // multi: proof / byte totals from pass 1 in dw[7] / dw[12], (spec, match) pairs in dw[20]
    IPCFP_CUDA(cudaStreamSynchronize(st));
    note_errors(hw);
    uint64_t n_exec = hw[3];
    const uint64_t M = hw[6];
    const uint64_t pass1_nodes = hw[4], pass1_bytes = hw[5];
    uint64_t n_proofs = hw[7], n_bytes = hw[12];
    const uint64_t n_pairs = ms ? hw[20] : M;

    // ---- PASS 2
    std::unique_ptr<EventResultBox> box(new EventResultBox());
    memset(&box->r, 0, sizeof box->r);
    AsyncBuf<ipcfp_event_proof> d_proofs(n_proofs + 1, st);
    AsyncBuf<uint8_t> d_blob(n_bytes + 16, st);
    uint32_t* any_skip_dev = misc.p + 2;
    // multi: the (spec, match) pairs in spec-major order, their proofs and bytes, the exclusive scans, per-spec bounds
    const uint64_t stride = (M + 31) / 32 * 32;
    if (ms && K * stride >= 0xffffffffull) throw Error(IPCFP_ERR_UNSUPPORTED, "n_specs x matching receipts exceeds 2^32");
    AsyncBuf<uint32_t> pair_bits(ms ? K * stride / 32 + 8 : 0, st), pairs(ms ? n_pairs + 32 : 0, st), pcnt(ms ? n_pairs + 8 : 0, st),
        pnby(ms ? n_pairs + 8 : 0, st);
    AsyncBuf<uint64_t> pair_prefix(ms ? K * stride / 32 + 8 : 0, st), spec_bounds(ms ? 3 * (K + 1) : 0, st);
    if (ms && M) {
        pbase.alloc(n_pairs + 8, st); bbase.alloc(n_pairs + 8, st);
        AsyncBuf<uint64_t> scratch_p(scan_scratch_elems(std::max<uint64_t>(n_pairs, K * stride / 32)) + 64, st);
        pair_bits.zero();
        k_pair_bits<<<div_up(M, 128), 128, 0, st>>>(match_rel.p, spec_mask.p, M, stride, pair_bits.p); IPCFP_LAUNCH_CHECK();
        // the scans below take the same launches whatever their size (≤ 16.7 M entries), so the call's launches do not depend on K
        bitmap_to_indices(pair_bits.p, K * stride, pairs.p, (uint64_t*)(dw + 21), pair_prefix.p, scratch_p.p, st, true);
        k_pair_count<<<div_up(n_pairs, 128), 128, 0, st>>>(s->view, s->view_dev.p, d_mm, td.events_roots.p, match_rel.p, pairs.p, n_pairs, stride, pcnt.p,
                                                          pnby.p); IPCFP_LAUNCH_CHECK();
        exclusive_scan_u32(pcnt.p, pbase.p, n_pairs, (uint64_t*)(dw + 22), scratch_p.p, st, true);
        exclusive_scan_u32(pnby.p, bbase.p, n_pairs, (uint64_t*)(dw + 23), scratch_p.p, st, true);
        k_spec_bounds<<<1, IPCFP_MAX_EVENT_SPECS + 1, 0, st>>>(pairs.p, n_pairs, stride, pbase.p, bbase.p, n_proofs, n_bytes, K, spec_bounds.p); IPCFP_LAUNCH_CHECK();
        Pass2MultiArgs p2;
        p2.store = s->view; p2.store_dev = s->view_dev.p; p2.mm = d_mm; p2.events_roots = td.events_roots.p; p2.match_rel = match_rel.p;
        p2.spec_mask = spec_mask.p; p2.n_match = M; p2.receipts_root_blk = receipts_root_blk; p2.exec_cids = exec_raw.p; p2.exec_idx = exec_idx.p;
        p2.n_exec = n_exec_dev; p2.wbits = wbits.p; p2.err = dw; p2.pair_bits = pair_bits.p; p2.pair_prefix = pair_prefix.p; p2.stride = stride;
        p2.pair_cnt = pcnt.p; p2.proof_cur = pbase.p; p2.byte_cur = bbase.p; p2.proofs = d_proofs.p; p2.blob = d_blob.p; p2.any_skip = any_skip_dev;
        p2.per_warp = M <= 16384 ? 1 : 0;
        k_pass2_multi<<<div_up(p2.per_warp ? M * 32 : M, 128), 128, 0, st>>>(p2); IPCFP_LAUNCH_CHECK();
    } else if (M) {
        Pass2Args p2;
        p2.store = s->view; p2.store_dev = s->view_dev.p; p2.m_dev = d_matcher; p2.m = mh; p2.events_roots = td.events_roots.p; p2.lo = lo; p2.match_rel = match_rel.p; p2.n_match = M;
        p2.receipts_root_blk = receipts_root_blk; p2.exec_cids = exec_raw.p; p2.exec_idx = exec_idx.p; p2.n_exec = n_exec_dev;
        p2.wbits = wbits.p; p2.err = dw; p2.cnt = cnt.p; p2.proof_base = pbase.p; p2.byte_base = bbase.p;
        p2.proofs = d_proofs.p; p2.blob = d_blob.p; p2.any_skip = any_skip_dev; p2.resolve_msg = sharded ? 0 : 1;
        p2.per_warp = (M <= 16384 && !getenv("IPCFP_PASS2_PER_THREAD")) ? 1 : 0;
        k_pass2<<<div_up(p2.per_warp ? M * 32 : M, 128), 128, 0, st>>>(p2); IPCFP_LAUNCH_CHECK();
    }
    if (xch) {
        // pass 2 did not wait for the cross-shard exchange; now that both are done: the global n_exec, the raw positions of this rank's
        // matches, and exec.get(i) of events/generator.rs:244-246 for every match — it PRECEDES r_amt.get(i) in the reference, so at the
        // same receipt it outranks whatever pass 2 reported (code 0 sorts first in the error word)
        // (all of it on the EXCHANGE stream, behind the exchange: the engine stream goes on with the witness and never waits for a peer)
        cudaStream_t sx = xch->stream();
        xch->positions_for(sx, match_rel.p, M, n_exec_dev);
        IPCFP_CUDA(cudaMemsetAsync(dw + 19, 0xff, 8, sx));   // the check has its own word: it may have to be repeated (stale exchange)
        if (M) { k_check_exec<<<div_up(M, 128), 128, 0, sx>>>(match_rel.p, M, lo, n_exec_dev, dw + 19); IPCFP_LAUNCH_CHECK(); }
        publish_words_on(s, sx, dw + 19, 19, 1);
    }
    // blocks recorded by pass 2 (receipt paths + events AMTs of the matches): the late part of the witness
    wbuild.finish_enqueue(wbits.p);
    publish_words(s, 0, 20);
    publish_words_from(s, misc.p, 20, 2);   // misc[2] = any_skip (32-bit words 0..3 land in hw[20..21])
    IPCFP_CUDA(cudaStreamSynchronize(st));
    if (ms && hw[0] != IPCFP_NO_ERROR && (uint32_t)(hw[0] >> 56) == ST_PASS2) {
        // (spec, i) key of pass2_multi_item: spec 0's missing base-witness block comes after spec 0's pass-2 faults and before those of
        // every later spec (materialize ends each of the reference's calls)
        if ((hw[0] >> 48) & 0xff && missing_base && !skip_tx) throw Error(IPCFP_ERR_MISSING_BLOCK, "missing block (base witness CID not in the store)");
        hw[0] &= ~(0xffull << 48);
    }
    note_errors(hw);
    // base-witness CIDs (parent headers, child header, TxMeta) are only dereferenced by WitnessCollector::materialize
    // (common/witness.rs:43-56, events/generator.rs:104), i.e. AFTER every receipts-root / pass-1 / pass-2 failure
    if (!xch && missing_base && !skip_tx) throw Error(IPCFP_ERR_MISSING_BLOCK, "missing block (base witness CID not in the store)");
    const uint64_t mB = hw[10];
    const bool any_skip = ((const uint32_t*)(hw + 20))[2] != 0;
    IPCFP_CUDA(cudaEventRecord(s->ev[4], st));

    // ---- results to the host
    box->matching = PinnedArray(s->pool, (n_pairs + 1) * 8);
    box->proofs = PinnedArray(s->pool, (n_proofs + 1) * sizeof(ipcfp_event_proof));
    box->blob = PinnedArray(s->pool, n_bytes + 16);
    PinnedArray rel(s->pool, (M + 1) * 4);
    if (M) IPCFP_CUDA(cudaMemcpyAsync(rel.p, match_rel.p, M * 4, cudaMemcpyDeviceToHost, st));
    PinnedArray pairs_h, bounds_h;
    if (ms && M) {
        pairs_h = PinnedArray(s->pool, n_pairs * 4);
        bounds_h = PinnedArray(s->pool, 3 * (K + 1) * 8);
        IPCFP_CUDA(cudaMemcpyAsync(pairs_h.p, pairs.p, n_pairs * 4, cudaMemcpyDeviceToHost, st));
        IPCFP_CUDA(cudaMemcpyAsync(bounds_h.p, spec_bounds.p, 3 * (K + 1) * 8, cudaMemcpyDeviceToHost, st));
    }
    if (n_proofs && !xch) IPCFP_CUDA(cudaMemcpyAsync(box->proofs.p, d_proofs.p, n_proofs * sizeof(ipcfp_event_proof), cudaMemcpyDeviceToHost, st));
    if (n_bytes) IPCFP_CUDA(cudaMemcpyAsync(box->blob.p, d_blob.p, n_bytes, cudaMemcpyDeviceToHost, st));

    // ---- witness: late blocks, sort in Cid order, index arrays (engine stream; the sharded protocol's tail runs beside it)
    wbuild.finish_start(mB, hw[11], box->wit);
    uint8_t* union_dev = nullptr;
    if (xch) {
        cudaStream_t sx = xch->stream();
        // H2: how far did every shard get. All ranks continue or fail together, naming the same first error. (The host waits for its
        // peers here while its own GPU sorts the witness.)
        IPCFP_CUDA(cudaStreamSynchronize(sx));
        uint64_t pend_chk = hw[19];
        xch->agree_results(pend_tx, std::min(pend_err, pend_chk), missing_base && !skip_tx, n_proofs, hw[8] + mB, xch->host_word(300), xch_stale);
        if (xch->g_stale && xch->g_tx == IPCFP_NO_ERROR) {
            // some shard's early promise was wrong: its slice differs from what the running exchange used. Every shard repeats the
            // exchange with the slices as they really are (late H0), then the positions, the exec.get check and H2.
            xch->agree_slices(pend_tx, pend_err, nraw);
            if (xch->peers_ok) {
                xch->start_exchange(exec_raw.p, s->ev[9]);
                xch->positions_for(sx, match_rel.p, M, n_exec_dev);
                IPCFP_CUDA(cudaMemsetAsync(dw + 19, 0xff, 8, sx));
                if (M) { k_check_exec<<<div_up(M, 128), 128, 0, sx>>>(match_rel.p, M, lo, n_exec_dev, dw + 19); IPCFP_LAUNCH_CHECK(); }
                publish_words_on(s, sx, dw + 19, 19, 1);
                IPCFP_CUDA(cudaStreamSynchronize(sx));
                pend_chk = hw[19];
            }
            xch->agree_results(pend_tx, std::min(pend_err, pend_chk), missing_base && !skip_tx, n_proofs, hw[8] + mB, xch->host_word(300), false);
        }
        if (xch->g_tx != IPCFP_NO_ERROR || xch->g_err != IPCFP_NO_ERROR || xch->g_missing_base || xch->g_overflow) {
            wbuild.finish_join(box->wit);   // nothing of this call may be in flight when its buffers go
            throw_global(xch->g_tx, xch->g_err, xch->g_missing_base);
            throw Error(IPCFP_ERR_UNSUPPORTED, "execution-order exchange: bucket overflow (skewed CID hash distribution)");
        }
        n_exec = xch->host_word(301);
        // EventProof.message_cid = exec[exec_index], fetched from the shards that hold them (pass 2 is complete: the host synchronised on it)
        xch->fetch_and_patch(sx, d_proofs.p, n_proofs);
        if (n_proofs) IPCFP_CUDA(cudaMemcpyAsync(box->proofs.p, d_proofs.p, n_proofs * sizeof(ipcfp_event_proof), cudaMemcpyDeviceToHost, sx));
        // union of the shards' witness CID sets as soon as this shard's sorted list exists (event after k_witness_emit), on its own
        // stream and communicator: it runs beside the message-CID fetch
        cudaStream_t sw = xch->union_stream();
        IPCFP_CUDA(cudaStreamWaitEvent(sw, s->ev[6], 0));
        if (flags & IPCFP_SHARDED_UNION_FULL) {
            xch->witness_union(sw, box->wit.cids_dev.p, box->wit.n, &union_dev, (uint64_t*)(dw + 18));
            publish_words_on(s, sw, dw + 18, 18, 1);
        } else xch->witness_union_partitioned(sw, box->wit.cids_dev.p, box->wit.n, xch->union_piece_cap(false), &union_dev, 320);   // [size, overflow] per rank → hw[320 ..)
    }
    wbuild.finish_join(box->wit);
    if (xch) {
        IPCFP_CUDA(cudaStreamSynchronize(xch->stream()));
        IPCFP_CUDA(cudaStreamSynchronize(xch->union_stream()));
        if (!(flags & IPCFP_SHARDED_UNION_FULL)) {
            bool overflow = false;
            for (uint32_t q = 0; q < world; q++) overflow |= hw[320 + 2 * q + 1] != 0;
            if (overflow) {   // a piece did not fit its slot on some rank (every rank sees the same words): once more with slots that cannot overflow
                xch->witness_union_partitioned(xch->union_stream(), box->wit.cids_dev.p, box->wit.n, xch->union_piece_cap(true), &union_dev, 320);
                IPCFP_CUDA(cudaStreamSynchronize(xch->union_stream()));
            }
        }
    }
    IPCFP_CUDA(cudaEventRecord(s->ev[5], st));
    IPCFP_CUDA(cudaStreamSynchronize(st));
    if (ms) {
        // spec k's part of matching_indices: its pairs, in receipt order; of proofs: [proof_off[k], proof_off[k + 1])
        uint64_t* mo = box->matching.as<uint64_t>();
        const uint32_t* rp = rel.as<uint32_t>();
        const uint32_t* pp = pairs_h.as<uint32_t>();
        for (uint64_t q = 0; q < n_pairs; q++) mo[q] = rp[pp[q] % stride];
        const uint64_t* bh = bounds_h.as<uint64_t>();
        for (uint32_t k = 0; k <= K; k++) {
            ms->match_off[k] = M ? bh[k] : 0;
            ms->proof_off[k] = M ? bh[K + 1 + k] : 0;
        }
        if (any_skip) {   // receipts the AMT does not hold: compact every spec's part
            ipcfp_event_proof* pr = box->proofs.as<ipcfp_event_proof>();
            uint64_t w = 0;
            for (uint32_t k = 0; k < K; k++) {
                const uint64_t b = ms->proof_off[k], e = ms->proof_off[k + 1];
                ms->proof_off[k] = w;
                for (uint64_t j = b; j < e; j++) if (pr[j].exec_index != UINT64_MAX) pr[w++] = pr[j];
            }
            ms->proof_off[K] = n_proofs = w;
        }
    } else {
        uint64_t* mo = box->matching.as<uint64_t>();
        const uint32_t* rp = rel.as<uint32_t>();
        for (uint64_t k = 0; k < M; k++) mo[k] = lo + rp[k];
    }
    if (any_skip && !ms) {  // receipts the AMT does not hold (`continue` at :249-251): compact their reserved slots away
        ipcfp_event_proof* pp = box->proofs.as<ipcfp_event_proof>();
        uint64_t w = 0;
        for (uint64_t k = 0; k < n_proofs; k++) if (pp[k].exec_index != UINT64_MAX) pp[w++] = pp[k];
        n_proofs = w;
    }
    ipcfp_event_result& r = box->r;
    r.n_matching = n_pairs; r.matching_indices = box->matching.as<uint64_t>();
    r.n_proofs = n_proofs; r.proofs = box->proofs.as<ipcfp_event_proof>();
    r.data_blob = box->blob.as<uint8_t>(); r.data_blob_size = n_bytes;
    box->wit.fill(r.witness);
    r.n_exec = n_exec;
    float el;
    IPCFP_CUDA(cudaEventElapsedTime(&el, s->ev[0], s->ev[5])); r.ms_total = el;
    IPCFP_CUDA(cudaEventElapsedTime(&el, s->ev[1], s->ev[2])); r.ms_txamt = el;
    IPCFP_CUDA(cudaEventElapsedTime(&el, s->ev[2], s->ev[3])); r.ms_pass1 = el;
    IPCFP_CUDA(cudaEventElapsedTime(&el, s->ev[3], s->ev[4])); r.ms_pass2 = el;
    IPCFP_CUDA(cudaEventElapsedTime(&el, s->ev[4], s->ev[5])); r.ms_witness = el;
    r.pass1_bytes = pass1_bytes; r.pass1_nodes = pass1_nodes;
    r.shard_raw_total = nraw_total;
    if (sharded) { r.n_exec = 0; r.shard_exec_count = nraw; box->shard_exec = std::move(exec_raw); r.shard_exec_dev = box->shard_exec.p; }
    if (xch) {
        r.n_exec = n_exec;
        r.union_cids_dev = union_dev;
        if (flags & IPCFP_SHARDED_UNION_FULL) { r.n_union_cids = r.n_union_part = hw[18]; r.union_part_first = 0; }
        else {
            r.n_union_cids = 0;
            for (uint32_t q = 0; q < world; q++) { if (q == rank) r.union_part_first = r.n_union_cids; r.n_union_cids += hw[320 + 2 * q]; }
            r.n_union_part = hw[320 + 2 * rank];
        }
        r.total_matching = xch->M_total; r.total_proofs = xch->proofs_total;
        xch->timings(&r.ms_exchange, &r.ms_fetch, &r.ms_union);
        if (getenv("IPCFP_XCH_TRACE")) {
            float t[6]; char buf[384];
            const int evs[6] = {2, 3, 4, 6, 7, 5};   // walk+snapshot done, pass 1 done, pass 2 done, sorted CID list, 51 MB copy done, end
            for (int i = 0; i < 6; i++) cudaEventElapsedTime(&t[i], s->ev[0], s->ev[evs[i]]);
            const auto t_now = std::chrono::steady_clock::now();
            const double host_call = std::chrono::duration<double, std::milli>(t_now - t_enter).count();
            const double host_gap = std::chrono::duration<double, std::milli>(t_enter - t_last_exit).count();
            snprintf(buf, sizeof buf, "host: gap since last call %.3f, in call %.3f | walk %.3f pass1 %.3f pass2 %.3f sorted %.3f blobD2H %.3f end %.3f", host_gap, host_call,
                     t[0], t[1], t[2], t[3], t[4], t[5]);
            t_last_exit = std::chrono::steady_clock::now();
            xch->trace_timeline(s->ev[0], buf);
        }
        if (flags & IPCFP_SHARDED_UNION_TO_HOST) {
            box->union_host = PinnedArray(s->pool, r.n_union_part * 38 + 64);
            if (r.n_union_part) IPCFP_CUDA(cudaMemcpyAsync(box->union_host.p, union_dev, r.n_union_part * 38, cudaMemcpyDeviceToHost, st));
            IPCFP_CUDA(cudaStreamSynchronize(st));
            r.union_cids = box->union_host.as<uint8_t>();
        }
    }
    return &box.release()->r;
}

void event_result_free(ipcfp_event_result* r) { delete reinterpret_cast<EventResultBox*>(r); }

void witness_cids_to_device(const ipcfp_event_result* r, void* dev_ptr, uint64_t cap, uint64_t* n) {
    uint64_t m = r->witness.n_blocks;
    if (m > cap) throw Error(IPCFP_ERR_INVALID_ARG, "device buffer too small for the witness CID list");
    const EventResultBox* box = reinterpret_cast<const EventResultBox*>(r);
    if (m) {
        if (box->wit.cids_dev.p) IPCFP_CUDA(cudaMemcpy(dev_ptr, box->wit.cids_dev.p, m * 38, cudaMemcpyDeviceToDevice));
        else IPCFP_CUDA(cudaMemcpy(dev_ptr, r->witness.cids, m * 38, cudaMemcpyHostToDevice));
    }
    *n = m;
}

}  // namespace ipcfp
