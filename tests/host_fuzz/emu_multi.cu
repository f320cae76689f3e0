// emu_multi.cu — the multi-spec event path (ipcfp_generate_event_proof_multi) executed ON THE CPU (TEST INFRASTRUCTURE, no GPU).
//
// The per-item device code of the multi-spec call, compiled for the host from the product headers and driven item by item:
//   pass 1 per receipt          pass1_multi_lookup + pass1_multi_decode (event_spec_mask, node_events_multi, walk_events_multi)
//   (spec, match) pairs          spec-major pair list as k_pair_bits + compaction build it, pair_count_item per pair
//   pass 2 per matching receipt  pass2_multi_item (receipts_get, ONE walk_events_multi<EMIT> for every spec of the receipt)
//   error order                  the (spec, i) key of pass 2, spec 0's missing base witness between spec 0's and spec 1's faults
// The setup, message-AMT walk and dedup are emu_events.cu's (included below); they are the single call's code.
// Checked against `oracle_generate_proof_bundle` with the same event specs: per-spec matching receipts, every EventProof field, the
// union witness, n_exec — and, with a block mutated under its CID or missing, the same (status, index). Half of the mutations hit a
// block only a later spec's matches reach.
//
//   nvcc -std=c++17 -O2 -o emu_multi tests/host_fuzz/emu_multi.cu oracle/oracle.cpp synth/synth.cpp -lpthread && ./emu_multi
#define main emu_events_main
#include "emu_events.cu"
#undef main

struct MultiOutcome {
    int status = IPCFP_OK;
    uint64_t index = UINT64_MAX;
    std::vector<std::vector<uint64_t>> matching;
    std::vector<std::vector<ProofRec>> proofs;
    std::set<std::string> witness;
    uint64_t n_exec = 0;
};

struct Spec { std::string sig, t1; bool has_actor; uint64_t actor; };

static ProofRec rec_of(const ipcfp_event_proof& q, const uint8_t* blob) {
    ProofRec pr;
    pr.exec_index = q.exec_index; pr.event_index = q.event_index; pr.emitter = q.emitter;
    pr.topics.assign((const char*)blob + q.topics_off, 32ull * q.n_topics);
    pr.data.assign((const char*)blob + q.data_off, q.data_len);
    pr.msg.assign((const char*)q.message_cid, 38);
    return pr;
}

static void engine_multi(const Blocks& B, const ipcfp_tipset_desc& td, const std::vector<Spec>& specs, MultiOutcome& o) {
    const uint32_t K = (uint32_t)specs.size();
    HostStore hs(B.cids.data(), B.offs.data(), B.lens.data(), B.blob.data(), B.blob.size(), B.n);
    const StoreView& sv = hs.view;
    const uint32_t P = td.n_parents, namt = 2 * P;
    unsigned long long err = IPCFP_NO_ERROR, txerr = IPCFP_NO_ERROR;
    std::vector<uint32_t> wbits((B.n + 31) / 32 + 8, 0);
    // ---- k_setup (emu_events.cu's sequence)
    bool missing_base = false;
    auto base = [&](const uint8_t* cid) { int32_t b = store_lookup_host_cid(sv, cid); if (b < 0) missing_base = true; else witness_mark(wbits.data(), (uint32_t)b); };
    for (uint32_t b = 0; b < P; b++) base(td.parent_cids + 38 * b);
    base(td.child_cid); base(td.receipts_root);
    for (uint32_t b = 0; b < P; b++) base(td.parent_txmeta_cids + 38 * b);
    std::vector<uint32_t> heights(namt, 0), f_blk(namt, 0), f_meta(namt, AMT_SENTINEL);
    std::vector<uint64_t> counts(namt, 0);
    for (uint32_t b = 0; b < P; b++) {
        int32_t tb = store_lookup_host_cid(sv, td.parent_txmeta_cids + 38 * b);
        if (tb < 0) { report_tx_error(&txerr, 3 * b, 0, 31, DC_MISSING, 0); continue; }
        witness_mark(wbits.data(), (uint32_t)tb);
        uint32_t len;
        const uint8_t* p = store_block(sv, (uint32_t)tb, len);
        Rd r(p, len);
        rd_array_exact(r, 2);
        uint32_t c0 = rd_cid(r), c1 = rd_cid(r);
        rd_end(r);
        if (r.err) { report_tx_error(&txerr, 3 * b, 0, 31, DC_DECODE, r.err); continue; }
        for (uint32_t k = 0; k < 2; k++) {
            int32_t rb = store_lookup(sv, p + (k ? c1 : c0));
            if (rb < 0) { report_tx_error(&txerr, 3 * b + 1 + k, 0, 31, DC_MISSING, 0); break; }
            witness_mark(wbits.data(), (uint32_t)rb);
            uint32_t rl;
            const uint8_t* rp = store_block(sv, (uint32_t)rb, rl);
            Rd rr(rp, rl);
            uint32_t bw, h;
            uint64_t cnt;
            amt_root_begin(rr, 0, bw, h, cnt);
            if (rr.err) { report_tx_error(&txerr, 3 * b + 1 + k, 0, 31, DC_DECODE, rr.err); break; }
            const uint32_t amt = 2 * b + k;
            f_blk[amt] = (uint32_t)rb; f_meta[amt] = make_meta(amt, 1, h); heights[amt] = h; counts[amt] = cnt;
        }
    }
    uint32_t receipts_root_blk = 0;
    {
        int32_t rb = store_lookup_host_cid(sv, td.receipts_root);
        if (rb < 0) report_error(&err, ST_RECEIPTS_ROOT, 0, DC_MISSING, 0);
        else {
            witness_mark(wbits.data(), (uint32_t)rb);
            receipts_root_blk = (uint32_t)rb;
            uint32_t len;
            const uint8_t* p = store_block(sv, (uint32_t)rb, len);
            Rd r(p, len);
            uint32_t bw, h;
            uint64_t cnt;
            amt_root_begin(r, 0, bw, h, cnt);
            AmtNodeHdr hd;
            amt_node_begin(r, 3, hd);
            uint32_t nv = rd_array(r);
            for (uint32_t v = 0; v < nv && !r.err; v++) parse_receipt(r);
            amt_node_finish(r, hd, nv, h);
            if (r.err) report_error(&err, ST_RECEIPTS_ROOT, 0, DC_DECODE, r.err);
        }
    }
    // ---- message-AMT walk: the general walk gives the same list, recording and errors as the dense one (emu_events.cu checks both)
    std::vector<uint64_t> rlo(namt), rhi(namt);
    shard_amt_ranges(namt, counts.data(), false, 0, td.n_receipts, td.n_receipts, rlo.data(), rhi.data());
    std::vector<RawCid> vals;
    uint64_t nraw = 0;
    uint32_t last_round = 0;
    for (uint32_t k = 0; k < namt; k++) last_round = std::max(last_round, heights[k]);
    host_general_walk(sv, namt, f_blk, f_meta, last_round, rlo.data(), rhi.data(), 1, wbits.data(), &txerr, 4 * B.n + 1024, vals, nraw);
    if (txerr != IPCFP_NO_ERROR) { Outcome t; fail_tx_key(t, txerr); o.status = t.status; o.index = t.index; return; }
    if (err != IPCFP_NO_ERROR) { Outcome t; fail_key(t, err); o.status = t.status; o.index = t.index; return; }
    std::vector<uint32_t> exec_idx;
    {
        std::unordered_set<std::string> seen;
        for (uint64_t k = 0; k < nraw; k++) if (seen.insert(std::string((const char*)vals[k].w, 40)).second) exec_idx.push_back((uint32_t)k);
    }
    unsigned long long n_exec = exec_idx.size();
    o.n_exec = n_exec;
    // ---- the staged MultiMatcher; t0 as k_spec_keccak computes it (zero padded, 8-byte aligned signature)
    MultiMatcher mm;
    memset(&mm, 0, sizeof mm);
    mm.n = K;
    for (uint32_t k = 0; k < K; k++) {
        Matcher& m = mm.m[k];
        std::vector<uint64_t> padded(specs[k].sig.size() / 8 + 2, 0);
        memcpy(padded.data(), specs[k].sig.data(), specs[k].sig.size());
        Digest d; keccak256((const uint8_t*)padded.data(), (uint32_t)specs[k].sig.size(), d); memcpy(m.t0, d.w, 32);
        uint8_t t1[32]; memset(t1, 0, 32); memcpy(t1, specs[k].t1.data(), std::min<size_t>(32, specs[k].t1.size())); memcpy(m.t1, t1, 32);
        m.actor = specs[k].actor; m.has_actor = specs[k].has_actor ? 1 : 0;
    }
    // ---- pass 1
    const uint64_t N = td.n_receipts;
    std::vector<uint8_t> roots_padded(N * 38 + 64, 0);
    if (N) memcpy(roots_padded.data(), td.events_roots, N * 38);
    std::vector<uint64_t> spec_mask(N + 8, 0);
    std::vector<uint32_t> match_rel;
    unsigned long long stats[2] = {0, 0}, n_proofs = 0, n_bytes = 0, n_pairs = 0;
    Pass1MultiArgs a1;
    memset(&a1, 0, sizeof a1);
    a1.store = sv; a1.store_dev = &sv; a1.mm = &mm; a1.events_roots = roots_padded.data(); a1.has_root = td.has_events_root; a1.n = N;
    a1.spec_mask = spec_mask.data(); a1.err = &err; a1.stats = stats; a1.n_proofs = &n_proofs; a1.n_bytes = &n_bytes; a1.n_pairs = &n_pairs;
    for (uint64_t i = 0; i < N; i++) {
        const int32_t blk = pass1_multi_lookup(a1, i);
        if (blk < 0) continue;
        uint32_t len;
        const uint8_t* p = store_block(sv, (uint32_t)blk, len);
        WalkOut wo{0, 0, false};
        const uint64_t mask = pass1_multi_decode(a1, mm, i, (uint32_t)blk, p, len, wo);
        if (!mask) continue;
        spec_mask[i] = mask;
        match_rel.push_back((uint32_t)i);
        n_proofs += wo.nproofs; n_bytes += wo.nbytes; n_pairs += (uint64_t)__builtin_popcountll(mask);
    }
    if (err != IPCFP_NO_ERROR) { Outcome t; fail_key(t, err); o.status = t.status; o.index = t.index; return; }
    // ---- (spec, match) pairs, their counts, the spec-major scans
    const uint64_t M = match_rel.size(), stride = (M + 31) / 32 * 32;
    std::vector<uint32_t> pair_bits(K * stride / 32 + 8, 0), pairs;
    for (uint64_t t = 0; t < M; t++)
        for (uint32_t k = 0; k < K; k++) if (spec_mask[match_rel[t]] >> k & 1) pair_bits[(k * stride + t) >> 5] |= 1u << ((k * stride + t) & 31);
    std::vector<uint64_t> pair_prefix(pair_bits.size() + 1, 0);
    for (size_t w = 0; w < pair_bits.size(); w++) {
        pair_prefix[w + 1] = pair_prefix[w] + (uint64_t)__builtin_popcount(pair_bits[w]);
        for (uint32_t b = 0; b < 32; b++) if (pair_bits[w] >> b & 1) pairs.push_back((uint32_t)(w * 32 + b));
    }
    if (pairs.size() != n_pairs) { o.status = 99; return; }
    std::vector<uint32_t> pcnt(n_pairs + 1, 0), pnby(n_pairs + 1, 0);
    for (uint64_t q = 0; q < n_pairs; q++) pair_count_item(sv, &sv, &mm, roots_padded.data(), match_rel.data(), pairs.data(), stride, q, pcnt.data(), pnby.data());
    std::vector<uint64_t> pbase(n_pairs + 1, 0), bbase(n_pairs + 1, 0);
    uint64_t tp = 0, tb = 0;
    for (uint64_t q = 0; q < n_pairs; q++) { pbase[q] = tp; bbase[q] = tb; tp += pcnt[q]; tb += pnby[q]; }
    if (tp != n_proofs || tb != n_bytes) { o.status = 98; return; }   // pass 1's totals must agree with the per-pair counts
    std::vector<uint64_t> proof_start(K + 1, tp), match_start(K + 1, n_pairs);
    for (uint32_t k = 0; k <= K; k++) {
        const uint64_t q = std::lower_bound(pairs.begin(), pairs.end(), (uint32_t)(k * stride)) - pairs.begin();
        match_start[k] = q;
        proof_start[k] = q < n_pairs ? pbase[q] : tp;
    }
    // ---- pass 2
    std::vector<ipcfp_event_proof> proofs(n_proofs + 1);
    std::vector<uint8_t> blob(n_bytes + 16);
    uint32_t any_skip = 0;
    Pass2MultiArgs a2;
    memset(&a2, 0, sizeof a2);
    a2.store = sv; a2.store_dev = &sv; a2.mm = &mm; a2.events_roots = roots_padded.data(); a2.match_rel = match_rel.data(); a2.spec_mask = spec_mask.data();
    a2.n_match = M; a2.receipts_root_blk = receipts_root_blk; a2.exec_cids = vals.data(); a2.exec_idx = exec_idx.data(); a2.n_exec = &n_exec;
    a2.wbits = wbits.data(); a2.err = &err; a2.pair_bits = pair_bits.data(); a2.pair_prefix = pair_prefix.data(); a2.stride = stride;
    a2.pair_cnt = pcnt.data(); a2.proof_cur = pbase.data(); a2.byte_cur = bbase.data(); a2.proofs = proofs.data(); a2.blob = blob.data(); a2.any_skip = &any_skip;
    for (uint64_t t = 0; t < M; t++) pass2_multi_item(a2, t);
    // ---- the host's error order (csrc/events.cu)
    if (err != IPCFP_NO_ERROR && (uint32_t)(err >> 56) == ST_PASS2) {
        if ((err >> 48) & 0xff && missing_base) { o.status = IPCFP_ERR_MISSING_BLOCK; o.index = UINT64_MAX; return; }
        err &= ~(0xffull << 48);
    }
    if (err != IPCFP_NO_ERROR) { Outcome t; fail_key(t, err); o.status = t.status; o.index = t.index; return; }
    if (missing_base) { o.status = IPCFP_ERR_MISSING_BLOCK; o.index = UINT64_MAX; return; }
    o.matching.assign(K, {});
    o.proofs.assign(K, {});
    for (uint32_t k = 0; k < K; k++) {
        for (uint64_t q = match_start[k]; q < match_start[k + 1]; q++) o.matching[k].push_back(match_rel[pairs[q] % stride]);
        for (uint64_t j = proof_start[k]; j < proof_start[k + 1]; j++)
            if (proofs[j].exec_index != UINT64_MAX) o.proofs[k].push_back(rec_of(proofs[j], blob.data()));
    }
    for (uint64_t i = 0; i < B.n; i++) if (wbits[i >> 5] >> (i & 31) & 1) o.witness.insert(std::string((const char*)B.cids.data() + 38 * i, 38));
}

static void oracle_bundle(const Blocks& B, const ipcfp_tipset_desc& td, const std::vector<Spec>& specs, MultiOutcome& o,
                          std::vector<std::set<std::string>>* per_spec_witness = nullptr) {
    oracle_store* os = oracle_store_create(B.cids.data(), B.offs.data(), B.lens.data(), B.blob.data(), B.n);
    std::vector<ipcfp_event_spec> es(specs.size());
    for (size_t k = 0; k < specs.size(); k++) {
        memset(&es[k], 0, sizeof es[k]);
        es[k].event_signature = specs[k].sig.c_str(); es[k].topic_1 = specs[k].t1.c_str();
        es[k].has_actor_id_filter = specs[k].has_actor ? 1 : 0; es[k].actor_id_filter = specs[k].actor;
    }
    ipcfp_bundle* b = nullptr;
    o.status = (int)oracle_generate_proof_bundle(os, &td, nullptr, 0, es.data(), es.size(), &b);
    if (o.status != IPCFP_OK) o.index = oracle_last_error_index();
    else {
        for (uint64_t k = 0; k < b->n_event_results; k++) {
            const ipcfp_event_result* er = b->events[k];
            o.matching.emplace_back(er->matching_indices, er->matching_indices + er->n_matching);
            o.proofs.emplace_back();
            for (uint64_t j = 0; j < er->n_proofs; j++) o.proofs.back().push_back(rec_of(er->proofs[j], er->data_blob));
            if (per_spec_witness) {
                per_spec_witness->emplace_back();
                for (uint64_t j = 0; j < er->witness.n_blocks; j++) per_spec_witness->back().insert(std::string((const char*)er->witness.cids + 38 * j, 38));
            }
            o.n_exec = er->n_exec;
        }
        for (uint64_t j = 0; j < b->witness.n_blocks; j++) o.witness.insert(std::string((const char*)b->witness.cids + 38 * j, 38));
        oracle_bundle_free(b);
    }
    oracle_store_destroy(os);
}

static int compare_multi(const Blocks& B, const ipcfp_tipset_desc& td, const std::vector<Spec>& specs, uint64_t* n_ok, uint64_t* n_err,
                         std::vector<std::set<std::string>>* per_spec_witness = nullptr) {
    MultiOutcome e, o;
    engine_multi(B, td, specs, e);
    oracle_bundle(B, td, specs, o, per_spec_witness);
    if (e.status != o.status || (e.status != IPCFP_OK && e.index != o.index)) {
        fprintf(stderr, "EMU MISMATCH: engine status %d index %lld vs oracle bundle status %d index %lld\n", e.status, (long long)e.index, o.status, (long long)o.index);
        return 1;
    }
    if (e.status != IPCFP_OK) { (*n_err)++; return 0; }
    for (size_t k = 0; k < specs.size(); k++) {
        if (e.matching[k] != o.matching[k]) { fprintf(stderr, "EMU MISMATCH: spec %zu matching (%zu vs %zu)\n", k, e.matching[k].size(), o.matching[k].size()); return 1; }
        if (!(e.proofs[k] == o.proofs[k])) { fprintf(stderr, "EMU MISMATCH: spec %zu proofs (%zu vs %zu)\n", k, e.proofs[k].size(), o.proofs[k].size()); return 1; }
    }
    if (e.n_exec != o.n_exec) { fprintf(stderr, "EMU MISMATCH: n_exec\n"); return 1; }
    if (e.witness != o.witness) { fprintf(stderr, "EMU MISMATCH: union witness (%zu vs %zu)\n", e.witness.size(), o.witness.size()); return 1; }
    (*n_ok)++;
    return 0;
}

static std::string sig_of(uint32_t j) { return j == 0 ? "NewTopDownMessage(bytes32,uint256)" : "Other" + std::to_string(j) + "(bytes32,uint256)"; }

int main(int argc, char** argv) {
    uint64_t cases = argc > 1 ? strtoull(argv[1], nullptr, 10) : 10;
    uint64_t muts = argc > 2 ? strtoull(argv[2], nullptr, 10) : 40;
    rs = argc > 3 ? strtoull(argv[3], nullptr, 10) : 0x3A17ull;
    uint64_t n_ok = 0, n_err = 0, n_later = 0;
    for (uint64_t c = 0; c < cases; c++) {
        synth_params sp;
        synth_default_params(&sp);
        sp.seed = 9000 + c * 13 + (rs & 0xff);
        static const uint64_t sizes[] = {1, 8, 9, 40, 64, 65, 257, 700};
        sp.n_receipts = sizes[rnd() % 8];
        static const uint32_t evs[] = {1, 3, 8, 8, 40};
        sp.events_per_receipt = evs[rnd() % 5];
        sp.match_ppm = 1000u << (rnd() % 10);
        if (sp.match_ppm > 1000000) sp.match_ppm = 1000000;
        sp.has_actor_filter = (uint32_t)(rnd() % 2);
        sp.bw3_permille = (uint32_t)(rnd() % 1001);
        sp.case_a_permille = rnd() % 2 ? (uint32_t)(rnd() % 500) : 0;
        sp.malformed_permille = rnd() % 3 == 0 ? (uint32_t)(rnd() % 100) : 0;
        sp.null_root_permille = rnd() % 2 ? (uint32_t)(rnd() % 300) : 0;
        sp.same_topic1 = (uint32_t)(rnd() % 4 == 0);
        sp.n_parents = 1 + (uint32_t)(rnd() % 3);
        sp.dup_msgs = (uint32_t)(rnd() % 4);
        sp.with_state_tree = 0;
        sp.threads = 1;
        synth_tipset* ts = synth_build(&sp);
        Blocks B;
        B.n = synth_n_blocks(ts);
        B.cids.assign(synth_cids(ts), synth_cids(ts) + 38 * B.n);
        B.offs.assign(synth_offsets(ts), synth_offsets(ts) + B.n);
        B.lens.assign(synth_lengths(ts), synth_lengths(ts) + B.n);
        B.blob.assign(synth_blob(ts), synth_blob(ts) + synth_blob_size(ts));
        ipcfp_tipset_desc td;
        memset(&td, 0, sizeof td);
        td.parent_epoch = synth_parent_epoch(ts); td.child_epoch = synth_child_epoch(ts); td.n_parents = synth_n_parents(ts);
        td.parent_cids = synth_parent_cids(ts); td.parent_txmeta_cids = synth_parent_txmeta_cids(ts); td.child_cid = synth_child_cid(ts);
        td.receipts_root = synth_receipts_root(ts); td.child_parent_state_root = synth_parent_state_root(ts); td.n_receipts = synth_n_receipts(ts);
        td.events_roots = synth_events_roots(ts); td.has_events_root = synth_has_events_root(ts);
        const std::string t1 = synth_topic1(ts);
        const uint64_t actor = synth_target_actor(ts);
        // disjoint, overlapping and identical specs; with same_topic1 every event carries the target's topic 1
        std::vector<Spec> specs;
        const uint32_t K = 1 + (uint32_t)(rnd() % 6);
        for (uint32_t k = 0; k < K; k++) {
            const uint32_t kind = (uint32_t)(rnd() % 5);
            if (kind == 0) specs.push_back({sig_of(0), t1, true, actor});
            else if (kind == 1) specs.push_back({sig_of(0), t1, false, 0});
            else if (kind == 2 && k) specs.push_back(specs[rnd() % k]);
            else {
                const std::string topic = sp.same_topic1 ? t1 : "calib-subnet-" + std::to_string(rnd() % 16);
                specs.push_back({sig_of((uint32_t)(rnd() % 8)), topic, rnd() % 2 == 0, 1000 + rnd() % 16});
            }
        }
        std::vector<std::set<std::string>> wit;
        if (compare_multi(B, td, specs, &n_ok, &n_err, &wit)) { fprintf(stderr, "  (tipset %llu as built, %u specs)\n", (unsigned long long)c, K); return 1; }
        // mutation targets: blocks that only a later spec's matches reach (first choice), any witness block otherwise
        std::vector<uint32_t> later, any;
        for (uint64_t i = 0; i < B.n; i++) {
            const std::string cid((const char*)B.cids.data() + 38 * i, 38);
            bool in0 = !wit.empty() && wit[0].count(cid), inl = false, inany = in0;
            for (size_t k = 1; k < wit.size(); k++) if (wit[k].count(cid)) inl = inany = true;
            if (inl && !in0) later.push_back((uint32_t)i);
            if (inany) any.push_back((uint32_t)i);
        }
        for (uint64_t mi = 0; mi < muts && !any.empty(); mi++) {
            const bool use_later = !later.empty() && mi % 2 == 0;
            const uint32_t victim = use_later ? later[rnd() % later.size()] : any[rnd() % any.size()];
            Blocks M = B;
            std::vector<uint8_t> blk(B.blob.begin() + (long)B.offs[victim], B.blob.begin() + (long)B.offs[victim] + B.lens[victim]);
            const size_t at = rnd() % blk.size();
            switch (rnd() % 4) {
                case 0: blk[at] ^= (uint8_t)(1u << (rnd() % 8)); break;
                case 1: blk.erase(blk.begin() + (long)at); break;
                case 2: blk.insert(blk.begin() + (long)at, (uint8_t)rnd()); break;
                default: blk.resize(at); break;
            }
            if (blk.empty()) blk.push_back(0x80);
            while (M.blob.size() % 16) M.blob.push_back(0);
            M.offs[victim] = M.blob.size();
            M.lens[victim] = (uint32_t)blk.size();
            M.blob.insert(M.blob.end(), blk.begin(), blk.end());
            if (rnd() % 6 == 0) M.cids[38ull * victim + 20] ^= 0x5a;                     // the block is not there at all
            if (mi % 5 == 0) M.cids[38ull * any[0] + 21] ^= 0xa5;                         // and a second fault elsewhere (often a base-witness block)
            n_later += use_later;
            if (compare_multi(M, td, specs, &n_ok, &n_err)) {
                fprintf(stderr, "  (tipset %llu, %u specs, mutation %llu of block %u%s)\n", (unsigned long long)c, K, (unsigned long long)mi, victim,
                        use_later ? ", reached by a later spec only" : "");
                return 1;
            }
        }
        synth_free(ts);
    }
    printf("ok: multi-spec event path on the CPU == oracle bundle for %llu tipsets: %llu runs equal in every field, %llu runs failing "
           "identically, %llu mutations in blocks only a later spec reaches\n",
           (unsigned long long)cases, (unsigned long long)n_ok, (unsigned long long)n_err, (unsigned long long)n_later);
    return 0;
}
