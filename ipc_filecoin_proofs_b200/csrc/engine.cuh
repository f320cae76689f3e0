// engine.cuh — host-side objects of the engine (C++17), shared by the translation units.
#pragma once
#include <array>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "store.cuh"
#include "rawcid.cuh"

namespace ipcfp {

// Grow-only cache of pinned host buffers so result read-backs run at PCIe rate without paying
// cudaHostAlloc on every call.
// Pinned host buffers should live on the NUMA node the GPU's PCIe root hangs off: a D2H / H2D that crosses the socket
// interconnect loses bandwidth, and with one process per GPU on a two-socket box half of the ranks would otherwise land
// on the far socket. Best effort and silent: the node comes from sysfs, the preference is a thread-local mempolicy
// (MPOL_PREFERRED, so allocation never fails because of it) that lasts for the lifetime of this guard.
struct NumaPrefer {
    bool on = false;
    int old_mode = 0;
    unsigned long old_mask[16] = {};   // the caller's own policy (e.g. numactl) is put back afterwards
    explicit NumaPrefer(int device);
    ~NumaPrefer();
};

struct PinnedPool {
    struct Buf { void* p; size_t cap; };
    std::mutex mu;
    std::vector<Buf> free_list;
    ~PinnedPool();
    void* take(size_t bytes, size_t* cap_out);
    void give(void* p, size_t cap);
};
struct PinnedArray {
    std::shared_ptr<PinnedPool> pool;
    void* p = nullptr;
    size_t cap = 0;
    PinnedArray() {}
    PinnedArray(std::shared_ptr<PinnedPool> pl, size_t bytes) : pool(std::move(pl)) { p = pool->take(bytes ? bytes : 16, &cap); }
    PinnedArray(const PinnedArray&) = delete;
    PinnedArray& operator=(const PinnedArray&) = delete;
    PinnedArray(PinnedArray&& o) noexcept : pool(std::move(o.pool)), p(o.p), cap(o.cap) { o.p = nullptr; }
    PinnedArray& operator=(PinnedArray&& o) noexcept { release(); pool = std::move(o.pool); p = o.p; cap = o.cap; o.p = nullptr; return *this; }
    ~PinnedArray() { release(); }
    void release() { if (p && pool) pool->give(p, cap); p = nullptr; }
    template <class T> T* as() const { return (T*)p; }
};

struct Store {
    int device = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr;
    uint64_t n = 0, blob_size = 0;
    DevBuf<uint8_t> arena;
    DevBuf<uint64_t> offsets;
    DevBuf<uint32_t> lengths;
    DevBuf<Digest> digests;
    DevBuf<uint8_t> cls;
    DevBuf<uint64_t> table;
    DevBuf<BlockRec> recs;
    DevBuf<uint32_t> rank_of, block_at_rank;   // `Cid` Ord rank of every block and its inverse (witness bitmaps are indexed by rank)
    StoreView view{};
    DevBuf<StoreView> view_dev;   // device copy, for out-of-line device functions (keeps kernel params off the stack)
    std::vector<std::array<uint8_t, 6>> class_prefix;  // distinct CID prefixes in this store
    std::vector<uint32_t> class_rank;                  // rank of each class in `Cid` Ord
    uint64_t first_bad = UINT64_MAX;
    std::shared_ptr<PinnedPool> pool;
    // small persistent scratch
    DevBuf<unsigned long long> dev_words;  // [0] error word, [1..] counters
    PinnedBuf<uint64_t> host_words;
    PinnedArray stage;                     // pinned staging (from the process-wide pool) for small per-call uploads: spec, tipset CIDs, walk tables
    cudaEvent_t ev[10] = {};
    ~Store();
    void use() const { IPCFP_CUDA(cudaSetDevice(device)); }
};

// Device-resident copy of an ipcfp_tipset_desc (events roots etc.)
struct TipsetDev {
    int64_t parent_epoch = 0, child_epoch = 0;
    uint32_t n_parents = 0;
    std::vector<uint8_t> parent_cids, txmeta_cids;  // host copies (tiny)
    uint8_t child_cid[38] = {}, receipts_root[38] = {}, child_state_root[38] = {};
    bool has_state_root = false;
    uint64_t n_receipts = 0;
    DevBuf<uint8_t> events_roots;  // n*38
    DevBuf<uint8_t> has_root;      // n
};

struct ScopedStatus;  // capi.cu
struct Comm;          // parallel.cu: NCCL communicator pair + exchange scratch of one rank

void set_last_error(const std::string& msg, uint64_t index);
ipcfp_status status_from_devcode(uint32_t code);

// store.cu
Store* store_create(const uint8_t* cids, const uint64_t* offsets, const uint32_t* lengths, const uint8_t* blob, uint64_t blob_size,
                    uint64_t n, int device, uint32_t flags);
void store_get(Store* s, const uint8_t* cid, uint8_t* buf, uint32_t cap, uint32_t* len, int* found);
void hash_batch(int which, const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets, const uint32_t* lengths, uint64_t n, int device,
                uint8_t* out);
void mapping_slots(const uint8_t* keys32, const uint64_t* slot_indices, uint64_t n, int device, uint8_t* out);
void check_device(int device);
// counters dev_words[first, first+count) → host_words (same indices) through mapped host memory: a tiny kernel
// instead of a D2H copy, so the read-back never queues behind a large copy on the copy engine
void publish_words(Store* s, uint32_t first, uint32_t count);
void publish_words_from(Store* s, const void* src_dev, uint32_t dst_first, uint32_t n_words);
void publish_words_on(Store* s, cudaStream_t stream, const void* src_dev, uint32_t dst_first, uint32_t n_words);   // the same on another stream

// events.cu
void tipset_upload(Store* s, const ipcfp_tipset_desc* t, TipsetDev& td);
// the reconstructed execution order of a tipset on the device (reconstruct_execution_order, events/utils.rs:16-30): exec[i] = exec_raw[exec_idx[i]]
struct ExecOrderOut {
    uint64_t n_exec = 0, nraw = 0;
    AsyncBuf<RawCid> exec_raw;
    AsyncBuf<uint32_t> exec_idx;
};
// ipcfp_generate_event_proof_multi: n specs scanned together; the caller's offset arrays have n + 1 entries each
struct MultiSpecs {
    const ipcfp_event_spec* specs;
    uint32_t n;
    uint64_t* match_off;
    uint64_t* proof_off;
};
ipcfp_event_result* generate_event_proof(Store* s, const ipcfp_tipset_desc* t, TipsetDev& td, const ipcfp_event_spec* spec, uint32_t flags,
                                         bool sharded, uint64_t lo, uint64_t hi, uint32_t world, uint32_t rank, Comm* comm = nullptr,
                                         ExecOrderOut* exo = nullptr, const MultiSpecs* ms = nullptr);
// verify.cu — batched verifiers over a witness store
void verify_event_proofs(Store* s, const ipcfp_tipset_desc* t, const ipcfp_event_proof* proofs, uint64_t n, const uint8_t* data_blob, uint64_t blob_size,
                         const ipcfp_event_spec* filter, uint8_t* results);
void verify_storage_proofs(Store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_proof* proofs, uint64_t n, uint8_t* results);
void event_result_free(ipcfp_event_result* r);
void witness_cids_to_device(const ipcfp_event_result* r, void* dev_ptr, uint64_t cap, uint64_t* n);
void merge_witness_cids(int device, const void* gathered, const uint64_t* counts, uint32_t world, uint64_t cap, void* out, uint64_t cap_out,
                        uint64_t* n_out);

// parallel.cu — in-library cross-shard protocol over NCCL (one process per GPU)
void comm_unique_id(uint8_t* id128);
Comm* comm_init(const uint8_t* id128, uint32_t world, uint32_t rank, int device);
void comm_destroy(Comm* c);
uint32_t comm_world(const Comm* c);
uint32_t comm_rank(const Comm* c);
// One sharded generate_event_proof call's share of the protocol (see the banner in parallel.cu). generate_event_proof drives it:
//   agree_slices → start_exchange → positions_for → agree_results → fetch_and_patch → witness_union
struct ShardExchange {
    Comm* c;
    Store* s;
    uint64_t lo, hi;
    // H0
    std::vector<uint64_t> nseg_all;
    uint64_t nraw = 0, max_nseg = 0, pos0 = 0, nseg = 0;
    bool peers_ok = true;
    bool all_early = false;          // early H0: every shard promised its slice before its walk was over
    // X
    const RawCid* seg = nullptr;
    uint64_t cap = 0, nwords = 0;
    unsigned long long* n_exec_dev = nullptr;
    unsigned long long* overflow_dev = nullptr;
    // P / F
    uint64_t M = 0;
    const uint32_t* match_rel_dev = nullptr;
    // H0 / H2 (global values, identical on every rank)
    uint64_t g_tx = ~0ull, g_err = ~0ull;
    bool g_missing_base = false, g_overflow = false, g_stale = false;
    uint64_t M_max = 0, nw_max = 0, M_total = 0, proofs_total = 0;
    std::vector<uint64_t> nw_all;
    ShardExchange(Comm* comm, Store* store, uint64_t lo_, uint64_t hi_);
    void agree_early(bool can_promise, uint64_t planned_nseg, uint64_t nraw_total);
    void agree_slices(uint64_t tx_key, uint64_t err_key, uint64_t nseg_);
    void start_exchange(const void* seg_dev, cudaEvent_t seg_ready);
    void positions_for(cudaStream_t st, const uint32_t* match_rel, uint64_t n_match, unsigned long long* n_exec_out);
    void agree_results(uint64_t tx_key, uint64_t err_key, bool missing_base, uint64_t n_proofs, uint64_t n_witness, uint64_t exch_overflow, bool stale);
    void fetch_and_patch(cudaStream_t st, ipcfp_event_proof* proofs_dev, uint64_t n_proofs);
    void witness_union(cudaStream_t st, const uint8_t* cids_dev, uint64_t n_local, uint8_t** out_dev, uint64_t* n_out_dev_word);
    // the same union left distributed: this rank's partition (sorted) in *out_dev; every rank's [partition size, overflow flag] lands in
    // the store's mapped words [host_word_first, +2·world) with the next sync of `st`. Any overflow flag set: repeat with
    // union_piece_cap(true).
    uint64_t union_piece_cap(bool cannot_overflow) const;
    void witness_union_partitioned(cudaStream_t st, const uint8_t* cids_dev, uint64_t n_local, uint64_t cap, uint8_t** out_dev, uint32_t host_word_first);
    void timings(float* ms_exchange, float* ms_fetch, float* ms_union) const;   // after the call's final sync
    void trace_timeline(cudaEvent_t origin, const char* engine_part) const;
    cudaStream_t stream() const;            // the exchange stream
    cudaStream_t union_stream() const;      // the witness union's own stream (its communicator is independent of the exchange's)
    uint64_t host_word(uint32_t i) const;   // the store's mapped words: 300 = exchange overflow flag, 301 = n_exec (valid after the sync that follows positions_for)
};
void exec_bucketize(int device, const void* seg, uint64_t nseg, uint64_t pos0, uint32_t world, uint64_t cap, void* send, uint64_t* counts_host);
void exec_dedup(int device, const void* recv, const uint64_t* counts, uint32_t world, uint64_t cap, uint64_t* dup_dev, uint64_t cap_out, uint64_t* n_dup);
void exec_fetch(int device, const void* seg, uint64_t nseg, uint64_t pos0, const uint64_t* req_dev, uint64_t n, void* out_dev);

// storage.cu
ipcfp_slot_result* read_storage_slots(Store* s, const uint8_t* root, const uint8_t* slots, uint64_t k);
void slot_result_free(ipcfp_slot_result* r);
ipcfp_storage_result* generate_storage_proofs(Store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_spec* specs, uint64_t n);
void storage_result_free(ipcfp_storage_result* r);

// witness.cu — materialise a witness bitmap into a sorted ipcfp_witness (host, pinned)
struct WitnessOut {
    PinnedArray cids, offsets, lengths, blob;
    PinnedArray sorted_idx;       // host copy of the block indices in Cid order (u32[n])
    AsyncBuf<uint8_t> cids_dev;   // the same sorted CIDs in device memory (n*38), for the multi-GPU union
    uint64_t n = 0, blob_size = 0;
    void fill(ipcfp_witness& w) const {
        w.n_blocks = n; w.cids = cids.as<uint8_t>(); w.offsets = offsets.as<uint64_t>(); w.lengths = lengths.as<uint32_t>();
        w.blob = blob.as<uint8_t>(); w.blob_size = blob_size;
    }
};
// Two-phase witness materialisation (see witness.cu): snapshot → start_copy → finish_enqueue → finish.
struct WitnessBuilder {
    Store* s;
    cudaStream_t st, st2;
    uint64_t nwords = 0, mA = 0, mB = 0, bytesA = 0, bytesB = 0, host_cap = 0;
    bool have_snapshot = false;
    bool by_ref = false;          // IPCFP_WITNESS_BY_REFERENCE: no block bytes are gathered or copied; offsets are the store's own
    AsyncBuf<uint32_t> idx, plen, bitsA, bitsB;
    AsyncBuf<uint64_t> offs, word_prefix, word_prefixB, scratch;
    AsyncBuf<uint8_t> dblobA, dblobB_keep;
    PinnedArray host_blob;
    explicit WitnessBuilder(Store* store);
    void snapshot(const uint32_t* wbits);        // enqueue; count → dev_words[8]
    // host knows the counts: gather in two parts (the first split_idx blocks = split_bytes bytes, then the rest) so that the D2H of
    // the first part is on the wire while the second is still being gathered
    void start_copy(uint64_t mA, uint64_t bytesA, uint64_t split_idx, uint64_t split_bytes);
    void finish_enqueue(const uint32_t* wbits);  // enqueue; late-block count → dev_words[10], their padded bytes → dev_words[11]
    // late blocks (mB of them, bytesB padded bytes: dev_words[10] and [11] after finish_enqueue), Cid-order index arrays, join
    void finish(uint64_t mB, uint64_t bytesB, WitnessOut& out, bool want_sorted_idx = false);
    void finish_start(uint64_t mB, uint64_t bytesB, WitnessOut& out, bool want_sorted_idx = false);   // … the same without the join: everything enqueued
    void finish_join(WitnessOut& out);                                              // … wait for both streams
};
void materialize_witness(Store* s, const uint32_t* wbits_dev, WitnessOut& out);
// ord[0..m) = the permutation that sorts the blocks idx[0..m) in `Cid` Ord (stable); runs on the store's stream (ingest: the ranks)
size_t sort_by_cid_ws_bytes(uint64_t m);
void sort_by_cid(Store* s, const uint32_t* idx_dev, uint32_t* ord, uint64_t m, void* workspace);

}  // namespace ipcfp
