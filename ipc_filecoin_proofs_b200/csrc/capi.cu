// capi.cu — the extern "C" surface declared in include/ipcfp.h.
#include <atomic>
#include <cstring>
#include <map>
#include <set>

#include "engine.cuh"
#include "prims.cuh"

namespace ipcfp {

static thread_local std::string g_last_error;
static thread_local uint64_t g_last_index = UINT64_MAX;
static std::atomic<uint64_t> g_launches{0};

void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
void set_last_error(const std::string& msg, uint64_t index) { g_last_error = msg; g_last_index = index; }

template <class F> static ipcfp_status guard(F f) {
    g_last_error.clear();
    g_last_index = UINT64_MAX;
    try { f(); return IPCFP_OK; }
    catch (const Error& e) { g_last_error = e.msg; g_last_index = e.index; return e.status; }
    catch (const std::bad_alloc&) { g_last_error = "out of host memory"; return IPCFP_ERR_INVALID_ARG; }
    catch (const std::exception& e) { g_last_error = e.what(); return IPCFP_ERR_INVALID_ARG; }
}

// ------------------------------------------------------------------------------------------ multi-GPU merge
// gathered: world segments of `cap` 38-byte CIDs, counts[r] valid in segment r. Sort + unique on the device.
struct SortCid { uint8_t b[38]; };
__global__ void k_merge_keys(const uint8_t* __restrict__ g, const uint64_t* __restrict__ seg_off, uint32_t world, uint64_t cap, uint64_t total,
                             uint32_t* keys, uint32_t* vals) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    uint32_t r = 0;
    while (r + 1 < world && i >= seg_off[r + 1]) r++;
    uint64_t src = (uint64_t)r * cap + (i - seg_off[r]);
    const uint8_t* c = g + 38 * src;
    keys[i] = ((uint32_t)c[6] << 24) | ((uint32_t)c[7] << 16) | ((uint32_t)c[8] << 8) | c[9];
    vals[i] = (uint32_t)src;
}
__device__ __forceinline__ int cid_cmp_raw(const uint8_t* a, const uint8_t* b) {
    for (int k = 0; k < 38; k++) if (a[k] != b[k]) return a[k] < b[k] ? -1 : 1;
    return 0;
}
__global__ void k_merge_tie_fix(const uint8_t* __restrict__ g, uint32_t* vals, const uint32_t* __restrict__ keys, uint64_t total) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    if (i > 0 && keys[i - 1] == keys[i]) return;
    if (i + 1 >= total || keys[i] != keys[i + 1]) return;
    uint64_t j = i + 1;
    while (j + 1 < total && keys[j + 1] == keys[i]) j++;
    for (uint64_t a = i + 1; a <= j; a++) {
        uint32_t v = vals[a];
        uint64_t b = a;
        while (b > i && cid_cmp_raw(g + 38ull * vals[b - 1], g + 38ull * v) > 0) { vals[b] = vals[b - 1]; b--; }
        vals[b] = v;
    }
}
__global__ void k_merge_unique_flags(const uint8_t* __restrict__ g, const uint32_t* __restrict__ vals, uint64_t total, uint32_t* bits) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool keep = false;
    if (i < total) keep = i == 0 || cid_cmp_raw(g + 38ull * vals[i - 1], g + 38ull * vals[i]) != 0;
    unsigned b = __ballot_sync(0xffffffffu, keep);
    if ((threadIdx.x & 31) == 0) bits[i >> 5] = b;
}
__global__ void k_merge_emit(const uint8_t* __restrict__ g, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ pos, uint64_t n,
                             uint8_t* out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* c = g + 38ull * vals[pos[i]];
    for (int k = 0; k < 38; k++) out[38 * i + k] = c[k];
}

void merge_witness_cids(int device, const void* gathered, const uint64_t* counts, uint32_t world, uint64_t cap, void* out, uint64_t cap_out,
                        uint64_t* n_out) {
    // NOTE: raw byte order == `Cid` Ord for CIDs sharing one prefix (the homogeneous Filecoin chain
    // case); stores with several CID prefixes must merge on the host (see DESIGN.md §6).
    check_device(device);
    std::vector<uint64_t> seg(world + 1, 0);
    for (uint32_t r = 0; r < world; r++) { if (counts[r] > cap) throw Error(IPCFP_ERR_INVALID_ARG, "count exceeds segment capacity"); seg[r + 1] = seg[r] + counts[r]; }
    uint64_t total = seg[world];
    *n_out = 0;
    if (!total) return;
    cudaStream_t st = nullptr;
    AsyncBuf<uint64_t> d_seg(world + 1, st);
    IPCFP_CUDA(cudaMemcpyAsync(d_seg.p, seg.data(), (world + 1) * 8, cudaMemcpyHostToDevice, st));
    AsyncBuf<uint32_t> keys(total, st), vals(total, st), ka(total, st), va(total, st), bits((total + 31) / 32 + 8, st), pos(total + 32, st);
    unsigned nb = radix_blocks(total);
    AsyncBuf<uint32_t> hist((size_t)256 * nb + 256, st);
    AsyncBuf<uint64_t> scan_tmp((size_t)256 * nb + 256, st), scratch(scan_scratch_elems(std::max<uint64_t>((uint64_t)256 * nb, total)) + 8, st),
        wp((total + 31) / 32 + 8, st), cnt(1, st);
    k_merge_keys<<<div_up(total, 256), 256, 0, st>>>((const uint8_t*)gathered, d_seg.p, world, cap, total, keys.p, vals.p); IPCFP_LAUNCH_CHECK();
    radix_sort_pairs(keys.p, vals.p, ka.p, va.p, total, 32, hist.p, scan_tmp.p, scratch.p, st);
    k_merge_tie_fix<<<div_up(total, 256), 256, 0, st>>>((const uint8_t*)gathered, vals.p, keys.p, total); IPCFP_LAUNCH_CHECK();
    k_merge_unique_flags<<<div_up((total + 31) / 32 * 32, 256), 256, 0, st>>>((const uint8_t*)gathered, vals.p, total, bits.p); IPCFP_LAUNCH_CHECK();
    bitmap_to_indices(bits.p, total, pos.p, cnt.p, wp.p, scratch.p, st);
    uint64_t n = 0;
    IPCFP_CUDA(cudaMemcpyAsync(&n, cnt.p, 8, cudaMemcpyDeviceToHost, st));
    IPCFP_CUDA(cudaStreamSynchronize(st));
    if (n > cap_out) throw Error(IPCFP_ERR_INVALID_ARG, "output buffer too small for the merged witness CID list");
    k_merge_emit<<<div_up(n, 256), 256, 0, st>>>((const uint8_t*)gathered, vals.p, pos.p, n, (uint8_t*)out); IPCFP_LAUNCH_CHECK();
    IPCFP_CUDA(cudaStreamSynchronize(st));
    *n_out = n;
}

// ------------------------------------------------------------------------------------------ bundle
struct BundleBox {
    ipcfp_bundle r;
    std::vector<ipcfp_event_result*> ev;
    std::vector<uint8_t> cids, blob;
    std::vector<uint64_t> offsets;
    std::vector<uint32_t> lengths;
};

}  // namespace ipcfp

using namespace ipcfp;

struct ipcfp_store { Store s; };

extern "C" {

const char* ipcfp_last_error(void) { return g_last_error.c_str(); }
uint64_t ipcfp_last_error_index(void) { return g_last_index; }
const char* ipcfp_version(void) {
    return "ipcfp-b200 0.2 (sm_100a): k_verify_cids k_hash_batch k_build_index sort_by_cid k_pass1_occ8 k_pass2 k_amt_dense k_amt_expand k_dedup "
           "k_storage_proofs k_read_slots k_verify_events k_verify_storage k_scan k_witness_copy k_witness_emit | sharded: k_xb_* k_exec_claim_seg "
           "k_exec_mark_dups k_select_positions k_fetch_positions k_part_pack k_merge_* (NCCL via dlopen)";
}
uint64_t ipcfp_kernel_launch_count(void) { return g_launches.load(); }

ipcfp_status ipcfp_host_alloc(size_t bytes, void** out) {
    return guard([&] {
        if (!out) throw Error(IPCFP_ERR_INVALID_ARG, "null out");
        int cnt = 0;
        if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { cudaGetLastError(); throw Error(IPCFP_ERR_NO_DEVICE, "no CUDA device"); }
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
        NumaPrefer numa(dev);   // pages of the caller's staging buffers next to the GPU they feed
        IPCFP_CUDA(cudaMallocHost(out, bytes ? bytes : 1));
    });
}
void ipcfp_host_free(void* p) { if (p) cudaFreeHost(p); }

ipcfp_status ipcfp_store_create(const uint8_t* cids, const uint64_t* offsets, const uint32_t* lengths, const uint8_t* blob, uint64_t blob_size,
                                uint64_t n_blocks, int device, uint32_t flags, ipcfp_store** out) {
    return guard([&] {
        if (!out) throw Error(IPCFP_ERR_INVALID_ARG, "null out");
        *out = nullptr;
        Store* s = store_create(cids, offsets, lengths, blob, blob_size, n_blocks, device, flags);
        *out = reinterpret_cast<ipcfp_store*>(s);
        if (s->first_bad != UINT64_MAX) throw Error(IPCFP_ERR_CID_MISMATCH, "blake2b-256(block) != CID digest", s->first_bad);
    });
}
void ipcfp_store_destroy(ipcfp_store* s) { delete reinterpret_cast<Store*>(s); }
uint64_t ipcfp_store_n_blocks(const ipcfp_store* s) { return s ? reinterpret_cast<const Store*>(s)->n : 0; }
uint64_t ipcfp_store_first_bad_block(const ipcfp_store* s) { return s ? reinterpret_cast<const Store*>(s)->first_bad : UINT64_MAX; }
ipcfp_status ipcfp_store_get(ipcfp_store* s, const uint8_t cid[IPCFP_CID_LEN], uint8_t* buf, uint32_t cap, uint32_t* len, int* found) {
    return guard([&] {
        if (!s || !cid || !found) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        store_get(reinterpret_cast<Store*>(s), cid, buf, cap, len, found);
    });
}
ipcfp_status ipcfp_store_has(ipcfp_store* s, const uint8_t cid[IPCFP_CID_LEN], int* found) {
    return guard([&] {
        if (!s || !cid || !found) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        uint32_t len;
        store_get(reinterpret_cast<Store*>(s), cid, nullptr, 0, &len, found);
    });
}

ipcfp_status ipcfp_blake2b256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets, const uint32_t* lengths, uint64_t n, int device,
                                    uint8_t* out) {
    return guard([&] { hash_batch(0, blob, blob_size, offsets, lengths, n, device, out); });
}
ipcfp_status ipcfp_keccak256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets, const uint32_t* lengths, uint64_t n, int device,
                                   uint8_t* out) {
    return guard([&] { hash_batch(1, blob, blob_size, offsets, lengths, n, device, out); });
}
ipcfp_status ipcfp_sha256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets, const uint32_t* lengths, uint64_t n, int device,
                                uint8_t* out) {
    return guard([&] { hash_batch(2, blob, blob_size, offsets, lengths, n, device, out); });
}
ipcfp_status ipcfp_compute_mapping_slots(const uint8_t* keys32, const uint64_t* slot_indices, uint64_t n, int device, uint8_t* out) {
    return guard([&] { mapping_slots(keys32, slot_indices, n, device, out); });
}

ipcfp_status ipcfp_generate_event_proof(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* spec, uint32_t flags,
                                        ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Store* st = reinterpret_cast<Store*>(s);
        TipsetDev td;
        tipset_upload(st, t, td);
        *out = generate_event_proof(st, t, td, spec, flags, false, 0, 0, 1, 0);
    });
}
ipcfp_status ipcfp_generate_event_proof_shard(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* spec, uint64_t lo, uint64_t hi,
                                              uint32_t world_size, uint32_t rank, uint32_t flags, ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Store* st = reinterpret_cast<Store*>(s);
        TipsetDev td;
        tipset_upload(st, t, td);
        *out = generate_event_proof(st, t, td, spec, flags, true, lo, hi, world_size, rank);
    });
}
void ipcfp_event_result_free(ipcfp_event_result* r) { if (r) event_result_free(r); }
ipcfp_status ipcfp_generate_event_proof_multi(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* specs, uint32_t n_specs, uint32_t flags,
                                              uint64_t* spec_match_offsets, uint64_t* spec_proof_offsets, ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Store* st = reinterpret_cast<Store*>(s);
        const MultiSpecs ms{specs, n_specs, spec_match_offsets, spec_proof_offsets};
        if (!specs || !spec_match_offsets || !spec_proof_offsets) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        if (n_specs == 0 || n_specs > IPCFP_MAX_EVENT_SPECS) throw Error(IPCFP_ERR_INVALID_ARG, "n_specs must be 1..IPCFP_MAX_EVENT_SPECS");
        TipsetDev td;
        tipset_upload(st, t, td);
        *out = generate_event_proof(st, t, td, nullptr, flags, false, 0, 0, 1, 0, nullptr, nullptr, &ms);
    });
}

ipcfp_status ipcfp_tipset_upload(ipcfp_store* s, const ipcfp_tipset_desc* t, ipcfp_tipset** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Store* st = reinterpret_cast<Store*>(s);
        std::unique_ptr<TipsetDev> td(new TipsetDev());
        tipset_upload(st, t, *td);
        IPCFP_CUDA(cudaStreamSynchronize(st->stream));
        *out = reinterpret_cast<ipcfp_tipset*>(td.release());
    });
}
void ipcfp_tipset_free(ipcfp_tipset* t) { delete reinterpret_cast<TipsetDev*>(t); }
ipcfp_status ipcfp_generate_event_proof_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec, uint32_t flags,
                                                 ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !t || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        *out = generate_event_proof(reinterpret_cast<Store*>(s), nullptr, *reinterpret_cast<TipsetDev*>(t), spec, flags, false, 0, 0, 1, 0);
    });
}
ipcfp_status ipcfp_generate_event_proof_multi_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* specs, uint32_t n_specs, uint32_t flags,
                                                       uint64_t* spec_match_offsets, uint64_t* spec_proof_offsets, ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !t || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        const MultiSpecs ms{specs, n_specs, spec_match_offsets, spec_proof_offsets};
        *out = generate_event_proof(reinterpret_cast<Store*>(s), nullptr, *reinterpret_cast<TipsetDev*>(t), nullptr, flags, false, 0, 0, 1, 0, nullptr,
                                    nullptr, &ms);
    });
}
ipcfp_status ipcfp_generate_event_proof_shard_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec, uint64_t lo, uint64_t hi,
                                                       uint32_t world_size, uint32_t rank, uint32_t flags, ipcfp_event_result** out) {
    return guard([&] {
        if (!s || !t || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        *out = generate_event_proof(reinterpret_cast<Store*>(s), nullptr, *reinterpret_cast<TipsetDev*>(t), spec, flags, true, lo, hi, world_size, rank);
    });
}
void* ipcfp_store_stream(ipcfp_store* s) { return s ? (void*)reinterpret_cast<Store*>(s)->stream : nullptr; }

ipcfp_status ipcfp_read_storage_slots(ipcfp_store* s, const uint8_t root[IPCFP_CID_LEN], const uint8_t* slots, uint64_t k, ipcfp_slot_result** out) {
    return guard([&] {
        if (!s || !out || !root || (k && !slots)) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        *out = read_storage_slots(reinterpret_cast<Store*>(s), root, slots, k);
    });
}
void ipcfp_slot_result_free(ipcfp_slot_result* r) { if (r) slot_result_free(r); }

ipcfp_status ipcfp_generate_storage_proofs(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_spec* specs, uint64_t n,
                                           ipcfp_storage_result** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        *out = generate_storage_proofs(reinterpret_cast<Store*>(s), t, specs, n);
    });
}
void ipcfp_storage_result_free(ipcfp_storage_result* r) { if (r) storage_result_free(r); }

// generate_proof_bundle (proofs/generator.rs:25-95): storage specs first, then event specs, then the
// BTreeSet<(Cid, Vec<u8>)> union of every proof's blocks. The union is a merge of already sorted,
// already materialised witness lists (host bookkeeping; no block is decoded or hashed here).
ipcfp_status ipcfp_generate_proof_bundle(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_spec* sspecs, uint64_t n_sspecs,
                                         const ipcfp_event_spec* especs, uint64_t n_especs, ipcfp_bundle** out) {
    return guard([&] {
        if (!s || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Store* st = reinterpret_cast<Store*>(s);
        std::unique_ptr<BundleBox> box(new BundleBox());
        memset(&box->r, 0, sizeof box->r);
        struct Cleanup { BundleBox* b; bool armed = true; ~Cleanup() { if (armed) { if (b->r.storage) storage_result_free(b->r.storage); for (auto* e : b->ev) event_result_free(e); } } } cl{box.get()};
        std::vector<const ipcfp_witness*> lists;
        if (n_sspecs) { box->r.storage = generate_storage_proofs(st, t, sspecs, n_sspecs); lists.push_back(&box->r.storage->witness); }
        if (n_especs) {
            TipsetDev td;
            tipset_upload(st, t, td);
            for (uint64_t i = 0; i < n_especs; i++) {
                box->ev.push_back(generate_event_proof(st, t, td, &especs[i], 0, false, 0, 0, 1, 0));
                lists.push_back(&box->ev.back()->witness);
            }
        }
        // k-way merge of sorted lists keyed by the store's CID order: reuse the order already
        // established on the device — equal CIDs are byte-identical, lists are individually sorted
        // by the same comparator, so a merge by (class rank, digest) bytes is exact.
        auto key_of = [&](const uint8_t* cid) {
            std::array<uint8_t, 39> k{};
            uint32_t rank = 0xff;
            for (size_t c = 0; c < st->class_prefix.size(); c++) if (!memcmp(cid, st->class_prefix[c].data(), 6)) rank = st->class_rank[c];
            k[0] = (uint8_t)rank;
            memcpy(k.data() + 1, cid + 6, 32);
            return k;
        };
        std::map<std::array<uint8_t, 39>, std::pair<const ipcfp_witness*, uint64_t>> uni;
        for (auto* w : lists) for (uint64_t i = 0; i < w->n_blocks; i++) uni.emplace(key_of(w->cids + 38 * i), std::make_pair(w, i));
        for (auto& kv : uni) {
            const ipcfp_witness* w = kv.second.first;
            uint64_t i = kv.second.second;
            box->cids.insert(box->cids.end(), w->cids + 38 * i, w->cids + 38 * i + 38);
            box->offsets.push_back(box->blob.size());
            box->lengths.push_back(w->lengths[i]);
            box->blob.insert(box->blob.end(), w->blob + w->offsets[i], w->blob + w->offsets[i] + w->lengths[i]);
        }
        box->r.n_event_results = box->ev.size();
        box->r.events = box->ev.data();
        box->r.witness.n_blocks = uni.size(); box->r.witness.cids = box->cids.data(); box->r.witness.offsets = box->offsets.data(); box->r.witness.lengths = box->lengths.data();
        box->r.witness.blob = box->blob.data(); box->r.witness.blob_size = box->blob.size();
        cl.armed = false;
        *out = &box.release()->r;
    });
}
void ipcfp_bundle_free(ipcfp_bundle* b) {
    if (!b) return;
    BundleBox* box = reinterpret_cast<BundleBox*>(b);
    if (box->r.storage) storage_result_free(box->r.storage);
    for (auto* e : box->ev) event_result_free(e);
    delete box;
}

ipcfp_status ipcfp_verify_event_proofs(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_proof* proofs, uint64_t n, const uint8_t* blob,
                                       uint64_t blob_size, const ipcfp_event_spec* filter, uint8_t* results) {
    return guard([&] {
        if (!s) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        verify_event_proofs(reinterpret_cast<Store*>(s), t, proofs, n, blob, blob_size, filter, results);
    });
}
ipcfp_status ipcfp_verify_storage_proofs(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_proof* proofs, uint64_t n, uint8_t* results) {
    return guard([&] {
        if (!s) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        verify_storage_proofs(reinterpret_cast<Store*>(s), t, proofs, n, results);
    });
}

ipcfp_status ipcfp_comm_unique_id(uint8_t id[IPCFP_COMM_ID_BYTES]) {
    return guard([&] {
        if (!id) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        comm_unique_id(id);
    });
}
ipcfp_status ipcfp_comm_init(const uint8_t id[IPCFP_COMM_ID_BYTES], uint32_t world_size, uint32_t rank, int device, ipcfp_comm** out) {
    return guard([&] {
        if (!id || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        *out = reinterpret_cast<ipcfp_comm*>(comm_init(id, world_size, rank, device));
    });
}
void ipcfp_comm_destroy(ipcfp_comm* c) { if (c) comm_destroy(reinterpret_cast<Comm*>(c)); }
ipcfp_status ipcfp_generate_event_proof_sharded(ipcfp_comm* c, ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec, const uint64_t* bounds,
                                                uint32_t flags, ipcfp_event_result** out) {
    return guard([&] {
        if (!c || !s || !t || !bounds || !out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        *out = nullptr;
        Comm* cm = reinterpret_cast<Comm*>(c);
        const uint32_t W = comm_world(cm), r = comm_rank(cm);
        TipsetDev& td = *reinterpret_cast<TipsetDev*>(t);
        for (uint32_t k = 0; k < W; k++) if (bounds[k] > bounds[k + 1]) throw Error(IPCFP_ERR_INVALID_ARG, "shard bounds must ascend");
        if (bounds[0] != 0 || bounds[W] != td.n_receipts) throw Error(IPCFP_ERR_INVALID_ARG, "shard bounds must cover [0, n_receipts)");
        *out = generate_event_proof(reinterpret_cast<Store*>(s), nullptr, td, spec, flags, true, bounds[r], bounds[r + 1], W, r, cm);
    });
}

ipcfp_status ipcfp_exec_bucketize(int device, const void* seg_dev, uint64_t nseg, uint64_t pos0, uint32_t world, uint64_t cap, void* send_dev,
                                  uint64_t* counts) {
    return guard([&] {
        if ((nseg && !seg_dev) || !send_dev || !counts) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        exec_bucketize(device, seg_dev, nseg, pos0, world, cap, send_dev, counts);
    });
}
ipcfp_status ipcfp_exec_dedup(int device, const void* recv_dev, const uint64_t* counts, uint32_t world, uint64_t cap, uint64_t* dup_pos_dev,
                              uint64_t cap_out, uint64_t* n_dup) {
    return guard([&] {
        if (!recv_dev || !counts || !dup_pos_dev || !n_dup) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        exec_dedup(device, recv_dev, counts, world, cap, dup_pos_dev, cap_out, n_dup);
    });
}
ipcfp_status ipcfp_exec_fetch(int device, const void* seg_dev, uint64_t nseg, uint64_t pos0, const uint64_t* req_pos_dev, uint64_t n_req,
                              void* out_dev) {
    return guard([&] {
        if ((nseg && !seg_dev) || (n_req && (!req_pos_dev || !out_dev))) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        exec_fetch(device, seg_dev, nseg, pos0, req_pos_dev, n_req, out_dev);
    });
}
ipcfp_status ipcfp_witness_cids_to_device(const ipcfp_event_result* r, void* dev_ptr, uint64_t cap_cids, uint64_t* n) {
    return guard([&] {
        if (!r || !dev_ptr || !n) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        witness_cids_to_device(r, dev_ptr, cap_cids, n);
    });
}
ipcfp_status ipcfp_merge_witness_cids(int device, const void* gathered_dev, const uint64_t* counts, uint32_t world, uint64_t cap, void* out_dev,
                                      uint64_t cap_out, uint64_t* n_out) {
    return guard([&] {
        if (!gathered_dev || !counts || !out_dev || !n_out) throw Error(IPCFP_ERR_INVALID_ARG, "null argument");
        merge_witness_cids(device, gathered_dev, counts, world, cap, out_dev, cap_out, n_out);
    });
}

}  // extern "C"
