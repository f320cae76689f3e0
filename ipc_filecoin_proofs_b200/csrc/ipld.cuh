// ipld.cuh — device-side decoders for the IPLD structures on the hot path:
//   AMT nodes  (fvm_ipld_amt 0.7 [UPSTREAM]: node = [bmap, [links], [values]];
//               root v0 = [height,count,node] bw 3; root v3 = [bit_width,height,count,node])
//   StampedEvent / ActorEvent / Entry + extract_evm_log (reference common/evm.rs:13-59)
//   Receipt 4-tuple, HAMT v3 nodes (fvm_ipld_hamt 0.10 [UPSTREAM]) and chain objects.
// One thread decodes one node; the decode contract is DESIGN.md §3.
#pragma once
#include "cbor.cuh"
#include "store.cuh"

namespace ipcfp {

// (actor_id, topic_0, topic_1) — EventMatcher of reference events/generator.rs:23-41
struct Matcher {
    uint64_t t0[4];   // keccak256(event_signature), little-endian word loads of the 32 bytes
    uint64_t t1[4];   // ascii_to_bytes32(topic_1)
    uint64_t actor;
    uint32_t has_actor;
};

__device__ __forceinline__ uint64_t pow_sat(uint32_t bw, uint32_t exp) {
    uint32_t s = bw * exp;
    return s >= 64 ? 0xFFFFFFFFFFFFFFFFull : (1ull << s);
}

__device__ __forceinline__ bool eq32(const uint8_t* p, const uint64_t w[4]) {
    if (load_u64_any(p) != w[0]) return false;
    return load_u64_any(p + 8) == w[1] && load_u64_any(p + 16) == w[2] && load_u64_any(p + 24) == w[3];
}

__device__ __forceinline__ bool cid38_equal(const uint8_t* a, const uint8_t* b) {
    bool eq = true;
    for (int k = 0; k < 38; k++) eq &= a[k] == b[k];
    return eq;
}

// ------------------------------------------------------------------ AMT node framing
// 256-bit bitmap as four scalars (no dynamically indexed arrays: those would live in local memory)
struct Bits256 {
    uint64_t b0, b1, b2, b3;
    __device__ __forceinline__ void clear() { b0 = b1 = b2 = b3 = 0; }
    __device__ __forceinline__ uint64_t word(uint32_t w) const { return w == 0 ? b0 : (w == 1 ? b1 : (w == 2 ? b2 : b3)); }
    __device__ __forceinline__ void or_byte(uint32_t i, uint32_t byte) {  // byte i (0..31), little-endian bit order
        uint64_t v = (uint64_t)byte << (8 * (i & 7));
        uint32_t w = i >> 3;
        b0 |= w == 0 ? v : 0; b1 |= w == 1 ? v : 0; b2 |= w == 2 ? v : 0; b3 |= w == 3 ? v : 0;
    }
    __device__ __forceinline__ uint32_t popc() const { return (uint32_t)(__popcll(b0) + __popcll(b1) + __popcll(b2) + __popcll(b3)); }
};
struct AmtNodeHdr {
    Bits256 bm;          // bit i of the node ↔ bm.word(i/64) >> (i%64)
    uint32_t pc;         // popcount
    uint32_t nl;         // number of links
    uint32_t links_off;  // offset of the first link item (each exactly 43 bytes)
};
// Reads `[bmap, [links…` up to and including the links array; links are validated.
__device__ __forceinline__ void amt_node_begin(Rd& r, uint32_t bw, AmtNodeHdr& h) {
    rd_array_exact(r, 3);
    uint32_t blen;
    uint32_t boff = rd_bytes(r, blen);
    uint32_t want = bw <= 3 ? 1u : (1u << (bw - 3));
    h.bm.clear();
    h.pc = 0;
    if (!r.err && blen != want) rd_fail(r, CE_AMT);
    if (!r.err) {
        for (uint32_t i = 0; i < blen; i++) h.bm.or_byte(i, r.p[boff + i]);
        uint32_t width = 1u << bw;
        if (width < 8 && (h.bm.b0 >> width)) rd_fail(r, CE_AMT);  // bit beyond the node width
        h.pc = h.bm.popc();
    }
    h.nl = rd_array(r);
    h.links_off = r.pos;
    for (uint32_t k = 0; k < h.nl && !r.err; k++) (void)rd_cid(r);
}
// Same as amt_node_begin up to the links array head, WITHOUT touching the links (callers that cannot read further
// than the first bytes of the node — the shared-memory ring of pass 1 — hand nodes with links to the full decoder).
__device__ __forceinline__ void amt_node_begin_head(Rd& r, uint32_t bw, AmtNodeHdr& h) {
    rd_array_exact(r, 3);
    uint32_t blen;
    uint32_t boff = rd_bytes(r, blen);
    uint32_t want = bw <= 3 ? 1u : (1u << (bw - 3));
    h.bm.clear();
    h.pc = 0;
    if (!r.err && blen != want) rd_fail(r, CE_AMT);
    if (!r.err) {
        for (uint32_t i = 0; i < blen; i++) h.bm.or_byte(i, r.p[boff + i]);
        uint32_t width = 1u << bw;
        if (width < 8 && (h.bm.b0 >> width)) rd_fail(r, CE_AMT);
        h.pc = h.bm.popc();
    }
    h.nl = rd_array(r);
    h.links_off = r.pos;
}
// after the values array has been consumed by the caller
__device__ __forceinline__ void amt_node_finish(Rd& r, const AmtNodeHdr& h, uint32_t nv, uint32_t height) {
    if (r.err) return;
    if (h.nl && nv) { rd_fail(r, CE_AMT); return; }
    if (h.nl) { if (height == 0 || h.pc != h.nl) rd_fail(r, CE_AMT); }
    else { if ((nv && height != 0) || h.pc != nv) rd_fail(r, CE_AMT); }
    if (!r.err) rd_end(r);
}
__device__ __forceinline__ bool bm_test(const Bits256& bm, uint32_t i) { return (bm.word(i >> 6) >> (i & 63)) & 1; }
__device__ __forceinline__ uint32_t bm_rank(const Bits256& bm, uint32_t i) {  // set bits below i
    uint32_t w = i >> 6, b = i & 63;
    uint32_t c = (w > 0 ? (uint32_t)__popcll(bm.b0) : 0) + (w > 1 ? (uint32_t)__popcll(bm.b1) : 0) + (w > 2 ? (uint32_t)__popcll(bm.b2) : 0);
    if (b) c += (uint32_t)__popcll(bm.word(w) & ((1ull << b) - 1));
    return c;
}
__device__ __forceinline__ uint32_t bm_select(const Bits256& bm, uint32_t k) {  // position of the k-th set bit
    for (uint32_t w = 0; w < 4; w++) {
        uint64_t x = bm.word(w);
        uint32_t c = (uint32_t)__popcll(x);
        if (k < c) {
            for (uint32_t j = 0; j < k; j++) x &= x - 1;
            return w * 64 + (uint32_t)(__ffsll((long long)x) - 1);
        }
        k -= c;
    }
    return 0xffffffffu;
}
// AMT roots. version 0: [height,count,node] (bw 3); version 3: [bw,height,count,node]
__device__ __forceinline__ void amt_root_begin(Rd& r, int version, uint32_t& bw, uint32_t& height, uint64_t& count) {
    if (version == 0) { rd_array_exact(r, 3); bw = 3; }
    else {
        rd_array_exact(r, 4);
        uint64_t b = rd_uint(r);
        if (!r.err && (b < 1 || b > 8)) rd_fail(r, CE_AMT);
        bw = r.err ? 3 : (uint32_t)b;
    }
    uint64_t h = rd_uint(r);
    if (!r.err && h * bw > 64) rd_fail(r, CE_AMT);
    height = r.err ? 0 : (uint32_t)h;
    count = rd_uint(r);
}

// ------------------------------------------------------------------ StampedEvent + extract_evm_log
struct EvLog {
    uint64_t emitter;
    uint32_t some;       // extract_evm_log returned Some
    uint32_t case_a;     // `topics`/`data` encoding
    uint32_t ntopics;
    uint32_t toff[4];    // Case B: offsets of t1..t4 values; Case A: toff[0] = offset of the topics blob
    uint32_t data_off, data_len;
};
// Per-event accumulator of the keys extract_evm_log looks at (last duplicate wins, evm.rs:14-17).
struct EvAcc {
    uint32_t have;    // bit0..3: t1..t4, bit4: d, bit5: topics, bit6: data
    uint32_t len_ok;  // bit0..3: tK value is exactly 32 bytes
    uint32_t t_off0, t_off1, t_off2, t_off3;
    uint32_t d_off, d_len, tp_off, tp_len, da_off, da_len;
    __device__ __forceinline__ void clear() { have = len_ok = 0; t_off0 = t_off1 = t_off2 = t_off3 = 0; d_off = d_len = tp_off = tp_len = da_off = da_len = 0; }
    __device__ __forceinline__ void topic(uint32_t idx, uint32_t voff, uint32_t vlen) {
        have |= 1u << idx;
        len_ok = vlen == 32 ? (len_ok | (1u << idx)) : (len_ok & ~(1u << idx));
        t_off0 = idx == 0 ? voff : t_off0; t_off1 = idx == 1 ? voff : t_off1;
        t_off2 = idx == 2 ? voff : t_off2; t_off3 = idx == 3 ? voff : t_off3;
    }
};
// extract_evm_log (common/evm.rs:13-59) over the accumulated keys: `topics` selects Case A (:20-30);
// Case B walks t1..t4, any present tK with len != 32 voids the log (:45-47), stops at the first gap
// (:50-52), no t1 ⇒ None (:54-56).
__device__ __forceinline__ void ev_finish(const EvAcc& a, EvLog& ev) {
    ev.some = 0; ev.case_a = 0; ev.ntopics = 0; ev.data_off = 0; ev.data_len = 0;
    ev.toff[0] = ev.toff[1] = ev.toff[2] = ev.toff[3] = 0;
    if (a.have & 32) {
        ev.case_a = 1;
        if (a.tp_len % 32 == 0) {
            ev.some = 1; ev.ntopics = a.tp_len / 32; ev.toff[0] = a.tp_off;
            if (a.have & 64) { ev.data_off = a.da_off; ev.data_len = a.da_len; }
        }
        return;
    }
    // number of leading present tK, and whether the first non-32-byte one comes before the first gap
    uint32_t present = a.have & 15, ok = a.len_ok & 15;
    uint32_t lead = present == 15 ? 4 : (uint32_t)(__ffs((int)(~present & 15)) - 1);  // t1..t(lead) present
    uint32_t lead_mask = (1u << lead) - 1;
    if (lead == 0 || (ok & lead_mask) != lead_mask) return;                              // no t1, or a bad length ⇒ None
    ev.some = 1; ev.ntopics = lead;
    ev.toff[0] = a.t_off0; ev.toff[1] = a.t_off1; ev.toff[2] = a.t_off2; ev.toff[3] = a.t_off3;
    if (a.have & 16) { ev.data_off = a.d_off; ev.data_len = a.d_len; }
}
// Generic strict decoder of one StampedEvent = [emitter, [[flags,key,codec,value]…]].
__device__ __forceinline__ void parse_stamped_event(Rd& r, EvLog& ev) {
    rd_array_exact(r, 2);
    ev.emitter = rd_uint(r);
    uint32_t ne = rd_array(r);
    EvAcc a;
    a.clear();
    for (uint32_t e = 0; e < ne && !r.err; e++) {
        rd_array_exact(r, 4);
        (void)rd_uint(r);
        uint32_t klen, vlen;
        uint32_t koff = rd_text(r, klen);
        (void)rd_uint(r);
        uint32_t voff = rd_bytes(r, vlen);
        if (r.err) break;
        const uint8_t* k = r.p + koff;
        if (klen == 2 && k[0] == 't') {
            uint32_t idx = (uint32_t)k[1] - (uint32_t)'1';
            if (idx < 4) a.topic(idx, voff, vlen);
        } else if (klen == 1 && k[0] == 'd') { a.have |= 16; a.d_off = voff; a.d_len = vlen; }
        else if (klen == 6 && bytes_eq(k, "topics", 6)) { a.have |= 32; a.tp_off = voff; a.tp_len = vlen; }
        else if (klen == 4 && bytes_eq(k, "data", 4)) { a.have |= 64; a.da_off = voff; a.da_len = vlen; }
    }
    ev_finish(a, ev);
    if (r.err) { ev.some = 0; ev.ntopics = 0; }
}

// Fast path: decodes a StampedEvent whose entries all have the canonical FEVM shape
//   84 <flags<24> <6x key> <codec: imm | 18 xx> <value: 40+n | 58 nn | 59 nnnn> value…
// with key ∈ {t1..t4, d, topics, data}, matching each entry against a 16-byte register window
// (three aligned 8-byte loads) instead of walking it byte by byte. Any deviation returns
// FAST_FAIL and the caller re-decodes the event with the generic strict parser, so results are
// identical by construction: the fast path only ever accepts encodings the strict parser
// accepts with the same meaning (minimal heads, ASCII keys, in-bounds values).
#define FAST_FAIL 0xffffffffu
__device__ __forceinline__ uint32_t win_byte(uint64_t w0, uint64_t w1, uint32_t k) {  // byte k (0..15) of the window
    uint64_t w = k < 8 ? w0 : w1;
    return (uint32_t)(w >> (8 * (k & 7))) & 0xffu;
}
// window source over global memory (the block arena)
template <int WINMODE = 0> struct GlobalWinT {   // WINMODE 1: two 16-byte loads per window instead of three 8-byte loads
    const uint8_t* p;
    __device__ __forceinline__ void load(uint32_t pos, uint64_t& w0, uint64_t& w1) { if (WINMODE) win_load16(p + pos, w0, w1); else win_load(p + pos, w0, w1); }
};
typedef GlobalWinT<0> GlobalWin;
template <class Win>
__device__ __forceinline__ uint32_t fast_stamped_event_t(Win& win, uint32_t pos, uint32_t n, EvLog& ev) {
    if (n - pos < 3) return FAST_FAIL;
    uint64_t w0, w1;
    win.load(pos, w0, w1);
    if ((w0 & 0xff) != 0x82) return FAST_FAIL;
    // emitter: a minimal uint head with ≤ 4 argument bytes (actor ids); 8-byte arguments take the strict parser
    uint32_t eb = (uint32_t)(w0 >> 8) & 0xff;
    if (eb >= 0x1b) return FAST_FAIL;                       // 8-byte argument, not major 0, or reserved ai
    uint32_t enb = eb < 24 ? 0 : (1u << (eb - 24));          // 0,1,2,4 argument bytes
    uint32_t be = __byte_perm((uint32_t)(w0 >> 16), 0, 0x0123);   // bytes 2..5, big-endian
    uint32_t earg = enb ? (be >> (32 - 8 * enb)) : eb;
    uint32_t emin = eb == 24 ? 24u : (eb == 25 ? 0x100u : (eb == 26 ? 0x10000u : 0u));
    if (earg < emin) return FAST_FAIL;                       // non-minimal → let the strict parser report it
    uint32_t hb = (uint32_t)(w0 >> (16 + 8 * enb)) & 0xffu;  // entries array head (enb ≤ 4 → byte ≤ 6)
    if ((hb & 0xe0) != 0x80 || (hb & 31) >= 24) return FAST_FAIL;
    uint32_t ne = hb & 31;
    uint32_t cur = pos + 3 + enb;
    if (cur > n) return FAST_FAIL;
    EvAcc a;
    a.clear();
    for (uint32_t e = 0; e < ne; e++) {
        if (n - cur < 5) return FAST_FAIL;
        win.load(cur, w0, w1);
        // the one shape almost every entry has — an indexed topic  84 fl 62 't' '1'..'4' 18 cc 58 LL  — is
        // recognised with constant masks on the window (all offsets static); anything else goes through the
        // general head decoder below. Both accept exactly the same encodings with the same (kind, voff, vlen).
        const uint32_t lo = (uint32_t)w0, hi = (uint32_t)(w0 >> 32), ll = (uint32_t)w1 & 0xffu;
        const uint32_t tidx = (hi & 0xffu) - (uint32_t)'1';
        const uint32_t fl8 = (lo >> 8) & 0xffu;
        bool canon = (lo & 0xffff00ffu) == 0x74620084u && fl8 < 24u && (hi & 0xff00ff00u) == 0x58001800u && tidx < 4u && ((hi >> 16) & 0xffu) >= 24u && ll >= 24u;
        uint32_t kind = tidx, vlen = ll, voff = cur + 9;
        // second static shape, the data entry  84 fl 61 'd' 18 cc <40+n | 58 nn | 59 nnnn>
        if ((lo & 0xffff00ffu) == 0x64610084u && fl8 < 24u && (hi & 0xffu) == 0x18u && ((hi >> 8) & 0xffu) >= 24u) {
            const uint32_t vb = (hi >> 16) & 0xffu, b7 = hi >> 24, l16 = (b7 << 8) | ll;
            kind = 4;
            if (vb - 0x40u < 0x18u) { vlen = vb - 0x40u; voff = cur + 7; canon = true; }
            else if (vb == 0x58u && b7 >= 24u) { vlen = b7; voff = cur + 8; canon = true; }
            else if (vb == 0x59u && l16 >= 256u) { vlen = l16; voff = cur + 9; canon = true; }
        }
        if (!canon) {
            uint32_t b0 = (uint32_t)w0 & 0xff, fl = (uint32_t)(w0 >> 8) & 0xff, th = (uint32_t)(w0 >> 16) & 0xff;
            if (b0 != 0x84 || fl >= 24) return FAST_FAIL;
            uint32_t klen = th - 0x60;                           // text head 0x61/0x62/0x64/0x66
            uint32_t k4 = (uint32_t)(w0 >> 24);                  // key bytes 0..3
            if (klen == 2) {
                uint32_t idx = ((k4 >> 8) & 0xff) - (uint32_t)'1';
                if ((k4 & 0xff) != 't' || idx >= 4) return FAST_FAIL;
                kind = idx;
            } else if (klen == 1) {
                if ((k4 & 0xff) != 'd') return FAST_FAIL;
                kind = 4;
            } else if (klen == 6) {
                uint64_t key = (w0 >> 24) | (w1 << 40);          // key bytes 0..5 in the low 48 bits
                if ((key & 0xffffffffffffull) != 0x736369706f74ull) return FAST_FAIL;  // "topics"
                kind = 5;
            } else if (klen == 4) {
                if (k4 != 0x61746164u) return FAST_FAIL;          // "data"
                kind = 6;
            } else return FAST_FAIL;
            uint32_t k = 3 + klen;                               // codec head position (≤ 9)
            uint32_t cb = win_byte(w0, w1, k);
            uint32_t clen;
            if (cb < 24) clen = 1;
            else if (cb == 24 && win_byte(w0, w1, k + 1) >= 24) clen = 2;
            else return FAST_FAIL;
            k += clen;                                           // value head position (≤ 11)
            uint32_t vb = win_byte(w0, w1, k);
            uint32_t vh;
            if (vb >= 0x40 && vb < 0x58) { vlen = vb - 0x40; vh = 1; }
            else if (vb == 0x58) { vlen = win_byte(w0, w1, k + 1); vh = 2; if (vlen < 24) return FAST_FAIL; }
            else if (vb == 0x59) { vlen = (win_byte(w0, w1, k + 1) << 8) | win_byte(w0, w1, k + 2); vh = 3; if (vlen < 256) return FAST_FAIL; }
            else return FAST_FAIL;
            voff = cur + k + vh;
        }
        if (voff > n || vlen > n - voff) return FAST_FAIL;
        if (kind < 4) a.topic(kind, voff, vlen);
        else if (kind == 4) { a.have |= 16; a.d_off = voff; a.d_len = vlen; }
        else if (kind == 5) { a.have |= 32; a.tp_off = voff; a.tp_len = vlen; }
        else { a.have |= 64; a.da_off = voff; a.da_len = vlen; }
        cur = voff + vlen;
    }
    ev.emitter = earg;
    ev_finish(a, ev);
    return cur;
}
template <int WINMODE = 0>
__device__ __forceinline__ uint32_t fast_stamped_event(const uint8_t* p, uint32_t pos, uint32_t n, EvLog& ev) {
    GlobalWinT<WINMODE> g{p};
    return fast_stamped_event_t(g, pos, n, ev);
}
// One StampedEvent at r.pos: fast path first, exact generic decoder on any deviation. The slow path
// works on private copies so that the caller's reader and EvLog stay in registers.
static __device__ __noinline__ uint32_t slow_stamped_event(const uint8_t* p, uint32_t pos, uint32_t n, EvLog* out, uint32_t* err) {
    Rd r2(p, n);
    r2.pos = pos;
    EvLog e2;
    parse_stamped_event(r2, e2);
    *out = e2;
    *err = r2.err;
    return r2.pos;
}
template <int WINMODE = 0>
__device__ __forceinline__ void decode_stamped_event(Rd& r, EvLog& ev) {
    if (r.err) { ev.some = 0; ev.ntopics = 0; ev.emitter = 0; return; }
    uint32_t np = fast_stamped_event<WINMODE>(r.p, r.pos, r.n, ev);
    if (np == FAST_FAIL) {
        EvLog e2;
        uint32_t err = 0;
        np = slow_stamped_event(r.p, r.pos, r.n, &e2, &err);
        ev = e2;
        if (err) { rd_fail(r, err); return; }
    }
    r.pos = np;
}
// actor filter (events/generator.rs:220-224) then matches_log (:38-40)
__device__ __forceinline__ bool event_matches(const uint8_t* p, const EvLog& ev, const Matcher& m) {
    if (m.has_actor && ev.emitter != m.actor) return false;
    if (!ev.some || ev.ntopics < 2) return false;
    uint32_t o0 = ev.toff[0], o1 = ev.case_a ? ev.toff[0] + 32 : ev.toff[1];
    return eq32(p + o0, m.t0) && eq32(p + o1, m.t1);
}
__device__ __forceinline__ uint32_t topic_offset(const EvLog& ev, uint32_t k) { return ev.case_a ? ev.toff[0] + 32 * k : ev.toff[k]; }

// Up to IPCFP_MAX_EVENT_SPECS EventMatchers tested together (ipcfp_generate_event_proof_multi): bit k of a mask is spec k.
struct MultiMatcher {
    Matcher m[IPCFP_MAX_EVENT_SPECS];   // first member: m[0] sits where the single-spec Matcher does
    uint32_t n;
};
// event_matches against every spec at once. The first 8 bytes of topics 0 and 1 are loaded once and screen the specs; a spec that
// passes the screen is compared in full.
__device__ __forceinline__ uint64_t event_spec_mask(const uint8_t* p, const EvLog& ev, const MultiMatcher& mm) {
    if (!ev.some || ev.ntopics < 2) return 0;
    const uint8_t* p0 = p + ev.toff[0];
    const uint8_t* p1 = p + (ev.case_a ? ev.toff[0] + 32 : ev.toff[1]);
    const uint64_t a = load_u64_any(p0), b = load_u64_any(p1);
    uint64_t mask = 0;
    for (uint32_t k = 0; k < mm.n; k++) {
        const Matcher& m = mm.m[k];
        if (m.t0[0] != a || m.t1[0] != b) continue;
        if (m.has_actor && ev.emitter != m.actor) continue;
        if (eq32(p0, m.t0) && eq32(p1, m.t1)) mask |= 1ull << k;
    }
    return mask;
}

// ------------------------------------------------------------------ Receipt = [exit_code, return_data, gas_used, events_root|null]
__device__ __forceinline__ void parse_receipt(Rd& r) {
    rd_array_exact(r, 4);
    uint64_t ec = rd_uint(r);
    if (!r.err && ec > 0xffffffffull) rd_fail(r, CE_RANGE);
    uint32_t l;
    (void)rd_bytes(r, l);
    (void)rd_uint(r);
    (void)rd_opt_cid(r);
}

// ------------------------------------------------------------------ HAMT (fvm_ipld_hamt v3 layout)
enum HamtValueKind { HV_ACTOR_STATE = 0, HV_U8VEC = 1 };
// value decoders: validate and remember where the value starts
__device__ __forceinline__ void parse_actor_state(Rd& r, uint32_t& state_cid_off) {
    rd_array_exact(r, 5);
    (void)rd_cid(r);
    state_cid_off = rd_cid(r);
    (void)rd_uint(r);
    uint32_t l;
    (void)rd_bytes(r, l);
    if (rd_peek_null(r)) r.pos++; else (void)rd_bytes(r, l);
}
// serde Vec<u8>: CBOR array of u8 (DESIGN.md §3); returns element count, elements start at r.pos after the head
__device__ __forceinline__ uint32_t parse_u8vec(Rd& r, uint32_t& first_elem_off) {
    uint32_t n = rd_array(r);
    first_elem_off = r.pos;
    for (uint32_t i = 0; i < n && !r.err; i++) { uint64_t x = rd_uint(r); if (!r.err && x > 255) rd_fail(r, CE_RANGE); }
    return n;
}

struct HamtHit {
    int32_t kind;          // 0 = None, 1 = value found, 2 = follow link
    uint32_t val_off;      // offset of the value item (kind 1)
    uint32_t link_off;     // offset of the 38 CID bytes (kind 2)
};
// Decodes a whole HAMT node (all pointers, all buckets, every value — like serde does) and resolves
// slot `idx` for `key`.
__device__ __forceinline__ void hamt_node_lookup(Rd& r, int vkind, uint32_t idx, const uint8_t* key, uint32_t keylen, HamtHit& hit) {
    hit.kind = 0; hit.val_off = 0; hit.link_off = 0;
    rd_array_exact(r, 2);
    uint32_t blen;
    uint32_t boff = rd_bytes(r, blen);
    if (!r.err && blen > 32) rd_fail(r, CE_HAMT);
    Bits256 bf;  // bf bit i ↔ child i; big-endian byte string, right aligned
    bf.clear();
    if (!r.err) for (uint32_t i = 0; i < blen; i++) bf.or_byte(i, r.p[boff + (blen - 1 - i)]);
    uint32_t np = rd_array(r);
    uint32_t pc = bf.popc();
    bool present = bm_test(bf, idx);
    uint32_t want = present ? bm_rank(bf, idx) : 0xffffffffu;
    for (uint32_t k = 0; k < np && !r.err; k++) {
        uint32_t mj = rd_peek_major(r);
        if (mj == 6) {
            uint32_t off = rd_cid(r);
            if (k == want && !r.err) { hit.kind = 2; hit.link_off = off; }
        } else if (mj == 4) {
            uint32_t nk = rd_array(r);
            for (uint32_t j = 0; j < nk && !r.err; j++) {
                rd_array_exact(r, 2);
                uint32_t kl;
                uint32_t ko = rd_bytes(r, kl);
                uint32_t voff = r.pos;
                if (vkind == HV_ACTOR_STATE) { uint32_t s; parse_actor_state(r, s); }
                else { uint32_t f; (void)parse_u8vec(r, f); }
                if (k == want && !r.err && hit.kind == 0 && kl == keylen) {
                    bool eq = true;
                    for (uint32_t b = 0; b < kl; b++) eq &= r.p[ko + b] == key[b];
                    if (eq) { hit.kind = 1; hit.val_off = voff; }
                }
            }
        } else if (!r.err) rd_fail(r, CE_HAMT);
    }
    if (!r.err) rd_end(r);
    if (!r.err && pc != np) rd_fail(r, CE_HAMT);
    if (r.err) hit.kind = 0;
}
// ---- fast HAMT node decode -------------------------------------------------------------------------------------------------
// hamt_node_lookup walks the node head by head with byte loads (≈ 20 dependent instructions per value ELEMENT — a Vec<u8> value is a
// CBOR array of small uints — i.e. ≈ 25 k instructions for a 1.5 KB node, 0.2 ms of one thread's time). This variant recognises the
// layout every node written by fvm_ipld_hamt has — short definite heads, 43-byte links, buckets of [bytes key, value] — with 8-byte
// window loads and skips value elements in registers (≈ 5 instructions each). It accepts ONLY what the strict decoder accepts, with the
// same hit; anything else returns false and the caller runs the strict decoder, which also names the error.
__device__ __forceinline__ bool skip_u8vec_fast(const uint8_t* p, uint32_t len, uint32_t& pos) {
    if (pos >= len) return false;
    uint64_t w0 = load_u64_any(p + pos);
    uint32_t b = (uint32_t)w0 & 0xff, n;
    if (b >= 0x80 && b < 0x98) { n = b - 0x80; pos += 1; }
    else if (b == 0x98) { n = (uint32_t)(w0 >> 8) & 0xff; if (n < 24 || len - pos < 2) return false; pos += 2; }
    else return false;                                   // longer arrays: strict path
    if (n > len - pos) return false;                     // (rd_array's bound: every element takes ≥ 1 byte)
    // One loop body for every lane (lanes of a warp walk different nodes: data-dependent branches would serialise them): a 16-byte
    // register window [base, base + 16) refilled every 8 bytes; an element is 1 byte (uint < 24) or `18 xx` with xx ≥ 24 (minimal
    // encoding); four two-byte elements in a row — the common run for random byte values — go in one step. Reads may run up to 24
    // bytes past `len` (every block buffer is padded by ≥ 32); a value that ends past the block is rejected after the loop.
    uint32_t base = pos;
    uint64_t w1 = load_u64_any(p + pos + 8);
    w0 = load_u64_any(p + pos);
    while (n) {
        uint32_t off = pos - base;
        if (off >= 8) { base = pos; w0 = load_u64_any(p + pos); w1 = load_u64_any(p + pos + 8); off = 0; }
        const uint32_t sh = 8 * off;                     // 0..56
        const uint64_t x = (w0 >> sh) | ((w1 << 1) << (63 - sh));
        const bool four = n >= 4 && (x & 0x00ff00ff00ff00ffull) == 0x0018001800180018ull &&
                          ((((x >> 8) & 0x00ff00ff00ff00ffull) + 0x00e800e800e800e8ull) & 0x0100010001000100ull) == 0x0100010001000100ull;
        const uint32_t e = (uint32_t)x & 0xff, e2 = (uint32_t)(x >> 8) & 0xff;
        if (four) { pos += 8; n -= 4; }
        else if (e < 0x18) { pos += 1; n -= 1; }
        else if (e == 0x18 && e2 >= 24) { pos += 2; n -= 1; }
        else return false;                               // > 255, non-minimal, another major type: the strict path decides
        if (pos > len) return false;
    }
    return true;
}
__device__ __forceinline__ bool hamt_node_lookup_fast(const uint8_t* p, uint32_t len, int vkind, uint32_t idx, const uint8_t* key, uint32_t keylen, HamtHit& hit) {
    hit.kind = 0; hit.val_off = 0; hit.link_off = 0;
    if (len < 3) return false;
    uint64_t w = load_u64_any(p);
    if ((w & 0xff) != 0x82) return false;
    uint32_t b1 = (uint32_t)(w >> 8) & 0xff, blen, boff;
    if (b1 >= 0x40 && b1 < 0x58) { blen = b1 - 0x40; boff = 2; }
    else if (b1 == 0x58) { blen = (uint32_t)(w >> 16) & 0xff; if (blen < 24 || blen > 32) return false; boff = 3; }
    else return false;
    if (boff + blen >= len) return false;
    Bits256 bf;
    bf.clear();
    for (uint32_t i = 0; i < blen; i++) bf.or_byte(i, p[boff + (blen - 1 - i)]);
    uint32_t pos = boff + blen;
    uint32_t hb = p[pos], np;
    if (hb >= 0x80 && hb < 0x98) { np = hb - 0x80; pos += 1; }
    else if (hb == 0x98) { if (len - pos < 2) return false; np = p[pos + 1]; if (np < 24) return false; pos += 2; }
    else return false;
    if (np > len - pos) return false;
    const uint32_t pc = bf.popc();
    const bool present = bm_test(bf, idx);
    const uint32_t want = present ? bm_rank(bf, idx) : 0xffffffffu;
    for (uint32_t k = 0; k < np; k++) {
        if (pos >= len) return false;
        w = load_u64_any(p + pos);
        const uint32_t b = (uint32_t)w & 0xff;
        if (b == 0xd8) {
            if ((w & 0xffffffffffffull) != 0x010027582ad8ull || len - pos < 43) return false;
            if (k == want) { hit.kind = 2; hit.link_off = pos + 5; }
            pos += 43;
        } else if (b >= 0x80 && b < 0x98) {
            const uint32_t nk = b - 0x80;
            pos += 1;
            if (nk > len - pos) return false;
            for (uint32_t j = 0; j < nk; j++) {
                if (len - pos < 3) return false;
                w = load_u64_any(p + pos);
                if ((w & 0xff) != 0x82) return false;
                const uint32_t kb = (uint32_t)(w >> 8) & 0xff;
                uint32_t kl, ko;
                if (kb >= 0x40 && kb < 0x58) { kl = kb - 0x40; ko = pos + 2; }
                else if (kb == 0x58) { kl = (uint32_t)(w >> 16) & 0xff; if (kl < 24) return false; ko = pos + 3; }
                else return false;
                if (ko > len || kl > len - ko) return false;
                pos = ko + kl;
                const uint32_t voff = pos;
                if (vkind == HV_U8VEC) { if (!skip_u8vec_fast(p, len, pos)) return false; }
                else {
                    Rd r(p, len);
                    r.pos = pos;
                    uint32_t so;
                    parse_actor_state(r, so);
                    if (r.err) return false;
                    pos = r.pos;
                }
                if (k == want && hit.kind == 0 && kl == keylen) {
                    bool eq = true;
                    for (uint32_t q = 0; q < kl; q++) eq &= p[ko + q] == key[q];
                    if (eq) { hit.kind = 1; hit.val_off = voff; }
                }
            }
        } else return false;
    }
    return pos == len && pc == np;
}

// bits [consumed, consumed+bw) of a SHA-256 digest given as 8 big-endian words, MSB first
__device__ __forceinline__ uint32_t hash_bits(const uint32_t h_be[8], uint32_t consumed, uint32_t bw) {
    uint32_t v = 0;
    for (uint32_t k = 0; k < bw; k++) {
        uint32_t bit = consumed + k;
        v = (v << 1) | ((h_be[bit >> 5] >> (31 - (bit & 31))) & 1u);
    }
    return v;
}

}  // namespace ipcfp
