/* ipcfp.h — C ABI of the B200-native witness-generation engine.
 *
 * Drop-in boundary for ONE path of consensus-shipyard/ipc-filecoin-proofs: the two-pass
 * receipt/event AMT scan and the HAMT storage-slot lookup. Every entry point cites the
 * reference interface it replaces (paths relative to the reference repo root). The header
 * is bindgen-ready: plain pointers and sizes, POD structs, no C++ or torch types.
 *
 * All compute behind these calls runs in hand-written sm_100a CUDA kernels. There is no
 * CPU implementation in this library: without a CUDA device every call fails with
 * IPCFP_ERR_NO_DEVICE.
 *
 * CIDs are 38-byte binary CIDv1 (`01 | codec | multihash code | 20 | digest[32]`; the
 * Filecoin chain form is `01 71 a0 e4 02 20 <blake2b-256>`), exactly the bytes behind the
 * strings `Cid::try_from(&str)` parses at src/proofs/common/witness.rs:60-63.
 *
 * Ownership: inputs are borrowed for the duration of the call. Outputs are owned by the
 * returned result object and released with the matching ipcfp_*_free. A store handle is
 * bound to one CUDA device; calls on one handle must be serialised by the caller.
 */
#ifndef IPCFP_H
#define IPCFP_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IPCFP_CID_LEN 38

typedef int32_t ipcfp_status;
enum {
    IPCFP_OK = 0,
    IPCFP_ERR_INVALID_ARG = -1,
    IPCFP_ERR_MISSING_BLOCK = -2,   /* anyhow!("missing ...") at witness.rs:47-50, storage/decode.rs:41-43, events/generator.rs:159-161 */
    IPCFP_ERR_DECODE = -3,          /* any serde / AMT / HAMT decode error bubbled by `?`                */
    IPCFP_ERR_CID_MISMATCH = -4,    /* IPCFP_STORE_VERIFY_CIDS: blake2b-256(block) != digest in its CID   */
    IPCFP_ERR_MISSING_EXEC = -5,    /* "Missing message at index" events/generator.rs:244-246             */
    IPCFP_ERR_CUDA = -6,
    IPCFP_ERR_NCCL = -7,
    IPCFP_ERR_STATE_ROOT_MISMATCH = -8, /* "ParentStateRoot mismatch" storage/generator.rs:93-99         */
    IPCFP_ERR_ACTOR_NOT_FOUND = -9,     /* "actor not found" common/decode.rs:39                         */
    IPCFP_ERR_NO_DEVICE = -10,
    IPCFP_ERR_UNSUPPORTED = -11
};

/* Thread-local description of the last failure on this thread ("" if none). */
const char* ipcfp_last_error(void);
/* Index attached to the last failure (receipt index / spec index / block index), or UINT64_MAX. */
uint64_t ipcfp_last_error_index(void);
/* Library version string and the list of kernels compiled in. */
const char* ipcfp_version(void);
/* Number of kernel launches issued by this library on the calling thread since load. */
uint64_t ipcfp_kernel_launch_count(void);

/* Pinned host memory for the flat block arrays (so ingest H2D copies run at PCIe rate). */
ipcfp_status ipcfp_host_alloc(size_t bytes, void** out);
void ipcfp_host_free(void* p);

/* ------------------------------------------------------------------------------------------
 * Block store — replaces the `fvm_ipld_blockstore::Blockstore` implementations the generators
 * are generic over (src/client/blockstore.rs:20-37, src/client/cached_blockstore.rs:53-85):
 * a device-resident arena of IPLD blocks with a CID hash index.
 * ------------------------------------------------------------------------------------------ */
typedef struct ipcfp_store ipcfp_store;

#define IPCFP_STORE_VERIFY_CIDS 0x1u /* Blake2b-256 every block on the GPU and compare with its CID */

/* cids: n*38 bytes; offsets[i]/lengths[i]: block i inside blob. Blocks are used in place at ANY offset / alignment
 * (every device read is an aligned load plus a byte shift). */
ipcfp_status ipcfp_store_create(const uint8_t* cids, const uint64_t* offsets, const uint32_t* lengths,
                                const uint8_t* blob, uint64_t blob_size, uint64_t n_blocks,
                                int device, uint32_t flags, ipcfp_store** out);
void ipcfp_store_destroy(ipcfp_store* s);
uint64_t ipcfp_store_n_blocks(const ipcfp_store* s);
/* Blockstore::get — copies the block into buf (cap bytes). *len receives the block length.
 * Unknown CID: returns IPCFP_OK with *found = 0 (the reference's Ok(None)). */
ipcfp_status ipcfp_store_get(ipcfp_store* s, const uint8_t cid[IPCFP_CID_LEN], uint8_t* buf, uint32_t cap,
                             uint32_t* len, int* found);
/* Blockstore::has */
ipcfp_status ipcfp_store_has(ipcfp_store* s, const uint8_t cid[IPCFP_CID_LEN], int* found);
/* Index of the first block whose CID digest did not match (after a CID_MISMATCH), else UINT64_MAX. */
uint64_t ipcfp_store_first_bad_block(const ipcfp_store* s);

/* ------------------------------------------------------------------------------------------
 * Batched hash primitives (unit parity of the kernels).
 * ------------------------------------------------------------------------------------------ */
/* out[i] = blake2b-256(blob[offsets[i] .. offsets[i]+lengths[i]))   (multihash-codetable Code::Blake2b256,
 * src/proofs/events/utils.rs:65) */
ipcfp_status ipcfp_blake2b256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets,
                                    const uint32_t* lengths, uint64_t n, int device, uint8_t* out /* n*32 */);
/* keccak256 (src/proofs/common/evm.rs:62-69, :81-88) */
ipcfp_status ipcfp_keccak256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets,
                                   const uint32_t* lengths, uint64_t n, int device, uint8_t* out /* n*32 */);
/* SHA-256 (fvm_ipld_hamt default key hasher) */
ipcfp_status ipcfp_sha256_batch(const uint8_t* blob, uint64_t blob_size, const uint64_t* offsets,
                                const uint32_t* lengths, uint64_t n, int device, uint8_t* out /* n*32 */);
/* compute_mapping_slot(key, slot_index) = keccak256(key32 || u256_be(slot_index))
 * (src/proofs/storage/utils.rs:5-12), batched. */
ipcfp_status ipcfp_compute_mapping_slots(const uint8_t* keys32 /* n*32 */, const uint64_t* slot_indices, uint64_t n,
                                         int device, uint8_t* out /* n*32 */);

/* ------------------------------------------------------------------------------------------
 * Inputs that came over RPC in the reference (src/client/types.rs:13-58).
 * ------------------------------------------------------------------------------------------ */
typedef struct ipcfp_tipset_desc {
    int64_t parent_epoch;                  /* parent.height                                   */
    int64_t child_epoch;                   /* child.height                                    */
    uint32_t n_parents;                    /* parent.cids.len() == parent.blocks.len()        */
    const uint8_t* parent_cids;            /* n_parents*38: parent.cids                       */
    const uint8_t* parent_txmeta_cids;     /* n_parents*38: parent.blocks[i].messages         */
    const uint8_t* child_cid;              /* 38: child.cids[0]                               */
    const uint8_t* receipts_root;          /* 38: child.blocks[0].parent_message_receipts     */
    const uint8_t* child_parent_state_root;/* 38: child.blocks[0].parent_state_root (JSON)    */
    uint64_t n_receipts;                   /* ChainGetParentReceipts(child) length            */
    const uint8_t* events_roots;           /* n_receipts*38: ApiReceipt.events_root           */
    const uint8_t* has_events_root;        /* n_receipts: 0 = None                            */
} ipcfp_tipset_desc;

/* EventProofSpec (src/proofs/generator.rs:18-22) */
typedef struct ipcfp_event_spec {
    const char* event_signature; /* e.g. "NewTopDownMessage(bytes32,uint256)" → topic0 = keccak256 */
    const char* topic_1;         /* ASCII, right-padded to 32 bytes (evm.rs:72-78)                  */
    uint8_t has_actor_id_filter;
    uint64_t actor_id_filter;
} ipcfp_event_spec;

/* StorageProofSpec (src/proofs/generator.rs:12-15) */
typedef struct ipcfp_storage_spec {
    uint64_t actor_id;
    uint8_t slot[32];
} ipcfp_storage_spec;

/* ------------------------------------------------------------------------------------------
 * Outputs.
 * ------------------------------------------------------------------------------------------ */
/* Vec<ProofBlock> in `Cid` Ord order (src/proofs/common/witness.rs:43-56, common/bundle.rs:11-18) */
typedef struct ipcfp_witness {
    uint64_t n_blocks;
    const uint8_t* cids;      /* n_blocks*38, sorted by (version, codec, multihash) */
    const uint64_t* offsets;  /* n_blocks: block i = blob[offsets[i] .. offsets[i]+lengths[i])   */
    const uint32_t* lengths;  /* n_blocks                                                        */
    const uint8_t* blob;      /* block bytes; blocks may sit in any order / with padding in here. NULL with IPCFP_WITNESS_BY_REFERENCE: offsets then index the blob given to ipcfp_store_create */
    uint64_t blob_size;
} ipcfp_witness;

/* EventProof + EventData (src/proofs/events/bundle.rs:6-23) minus the per-call constants
 * (epochs, parent tipset CIDs, child block CID) which the caller already holds. */
typedef struct ipcfp_event_proof {
    uint64_t exec_index;
    uint64_t event_index;
    uint64_t emitter;
    uint32_t n_topics;      /* ≤ 4 in Case B; Case A (`topics` key) may carry more — see data_off   */
    uint32_t data_len;
    uint64_t data_off;      /* into ipcfp_event_result.data_blob                                    */
    uint64_t topics_off;    /* into data_blob: n_topics*32 bytes                                    */
    uint8_t message_cid[IPCFP_CID_LEN];
    uint8_t _pad[2];
} ipcfp_event_proof;

typedef struct ipcfp_event_result {
    uint64_t n_matching;
    const uint64_t* matching_indices; /* pass-1 output (events/generator.rs:206-239), ascending */
    uint64_t n_proofs;
    const ipcfp_event_proof* proofs;  /* ordered by (exec_index, event_index)                  */
    const uint8_t* data_blob;
    uint64_t data_blob_size;
    ipcfp_witness witness;            /* EventProofBundle.blocks                                */
    uint64_t n_exec;                  /* length of the reconstructed execution order            */
    /* device-side timing of the last call, milliseconds (CUDA events on the engine stream) */
    float ms_total, ms_pass1, ms_pass2, ms_txamt, ms_witness;
    uint64_t pass1_bytes;             /* algorithmic bytes read by the pass-1 scan kernel       */
    uint64_t pass1_nodes;
    /* shard mode only (ipcfp_generate_event_proof_shard): this shard's slice of the concatenated message list,
     * in order, as 40-byte records {digest[32], prefix[6], 0, 0} in DEVICE memory (valid until the result is
     * freed; free results before destroying the store). proofs[].message_cid is left zero and n_exec is 0:
     * the execution order spans shards and is resolved by the caller (ipcfp_exec_* helpers). */
    const void* shard_exec_dev;
    uint64_t shard_exec_count;
    uint64_t shard_raw_total;         /* total length of the concatenated message list (all shards) */
    /* ipcfp_generate_event_proof_sharded only: proofs[].message_cid and n_exec are final (resolved across shards inside the
     * call). The union of ALL shards' witness CID sets (the BTreeSet union of src/proofs/common/witness.rs:24-40) has
     * n_union_cids entries in `Cid` order and is left DISTRIBUTED: this rank holds entries [union_part_first, union_part_first +
     * n_union_part) — the CIDs whose first two digest bytes fall into its 1/world share of the 65 536 buckets — so the
     * concatenation of the ranks' parts in rank order is the whole sorted set. With IPCFP_SHARDED_UNION_FULL every rank holds the
     * whole set instead (union_part_first = 0, n_union_part = n_union_cids). union_cids_dev: DEVICE memory, n_union_part*38 bytes,
     * valid until the next sharded call on the same communicator; union_cids: the same on the host with
     * IPCFP_SHARDED_UNION_TO_HOST. total_matching / total_proofs: summed over all shards. */
    const void* union_cids_dev;
    uint64_t n_union_cids;
    const uint8_t* union_cids;
    uint64_t total_matching;
    uint64_t total_proofs;
    float ms_exchange, ms_fetch, ms_union; /* device time of the execution-order exchange (its own stream, under pass 1), the message-CID fetch, the witness union */
    float _pad0;
    uint64_t union_part_first;
    uint64_t n_union_part;
} ipcfp_event_result;

typedef struct ipcfp_storage_proof {
    uint64_t actor_id;
    uint8_t actor_state_cid[IPCFP_CID_LEN];
    uint8_t storage_root[IPCFP_CID_LEN];
    uint8_t slot[32];
    uint8_t value[32];    /* left_pad_32(raw) (evm.rs:91-100); zero when absent */
    uint8_t found;        /* Hamt::get returned Some                            */
    uint8_t _pad[3];
    uint32_t raw_len;     /* length of the raw value                            */
} ipcfp_storage_proof;

typedef struct ipcfp_storage_result {
    uint64_t n_proofs;
    const ipcfp_storage_proof* proofs;
    ipcfp_witness witness;              /* union over all specs, sorted                          */
    const uint64_t* spec_witness_offsets; /* n_proofs+1                                          */
    const uint32_t* spec_witness_index;   /* per spec: indices into witness (its Vec<ProofBlock>) */
    float ms_total;
} ipcfp_storage_result;

typedef struct ipcfp_slot_result {
    uint64_t n;
    const uint8_t* found;      /* n                                        */
    const uint32_t* raw_len;   /* n                                        */
    const uint8_t* values;     /* n*32, left-padded                        */
    ipcfp_witness witness;     /* blocks touched by the lookups (recorder) */
    float ms_total;
    float ms_lookup;           /* device time of the lookup kernel alone (CUDA events on the engine stream)              */
    uint64_t lookup_nodes;     /* HAMT nodes decoded by the lookups                                                      */
    uint64_t lookup_bytes;     /* algorithmic bytes of the lookups: 32 per key + the bytes of every node on its path      */
} ipcfp_slot_result;

typedef struct ipcfp_bundle {
    ipcfp_storage_result* storage;  /* may be NULL */
    uint64_t n_event_results;
    ipcfp_event_result** events;    /* one per event spec */
    ipcfp_witness witness;          /* UnifiedProofBundle.blocks: BTreeSet<(Cid, data)> order */
} ipcfp_bundle;

/* ------------------------------------------------------------------------------------------
 * Entry points.
 * ------------------------------------------------------------------------------------------ */
#define IPCFP_SCAN_SKIP_TX_AMTS 0x1u  /* find_matching_events only: no record_transaction_amts / base witness;
                                         execution order still built                                          */
#define IPCFP_SHARDED_UNION_TO_HOST 0x2u /* ipcfp_generate_event_proof_sharded: also copy this rank's part of the merged witness CID list to the host */
/* Witness BY REFERENCE (all ipcfp_generate_event_proof* calls): the result's witness carries no block bytes. witness.blob is NULL,
 * blob_size 0, and offsets[i] / lengths[i] locate block i inside the blob the STORE WAS CREATED FROM (the caller's own host array,
 * which it still holds): cids / offsets / lengths arrive as usual, in `Cid` order. Saves copying ≈ 51 MB per 1 M receipts that the
 * host already has; WitnessCollector::materialize (src/proofs/common/witness.rs:43-56) becomes a gather over the caller's blocks. */
#define IPCFP_WITNESS_BY_REFERENCE 0x8u
#define IPCFP_SHARDED_UNION_FULL 0x4u    /* … every rank receives the WHOLE merged list (all-gather + merge of `world` lists on every rank) instead of its partition */

/* generate_event_proof (src/proofs/events/generator.rs:60-107): base witness, message-AMT
 * recording, execution order, two-pass scan (find_matching_events :180-307), materialise. */
ipcfp_status ipcfp_generate_event_proof(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* spec,
                                        uint32_t flags, ipcfp_event_result** out);
void ipcfp_event_result_free(ipcfp_event_result* r);

/* The event half of generate_proof_bundle (src/proofs/generator.rs:57-78) in ONE scan of the tipset for n_specs specs
 * (1 ≤ n_specs ≤ IPCFP_MAX_EVENT_SPECS): base witness, message-AMT walk and execution order once, one pass-1 launch that tests every
 * spec on every StampedEvent, pass 2 over the union of the specs' matches, and ONE witness: the BTreeSet union of the specs'
 * witnesses. With B = ipcfp_generate_proof_bundle(s, t, NULL, 0, specs, n_specs):
 *   matching_indices  the concatenation in spec order of B.events[k].matching_indices; spec k's part is
 *                     [spec_match_offsets[k], spec_match_offsets[k+1]), n_matching the total
 *   proofs            the concatenation in spec order of B.events[k].proofs; spec k's part is [spec_proof_offsets[k], spec_proof_offsets[k+1])
 *   data_blob         the concatenation in spec order of the specs' data blobs; topics_off / data_off point into it
 *   witness, n_exec   B.witness byte for byte; the single call's n_exec
 * Identical specs give their proofs twice; a spec that matches nothing has an empty part. Flags as for ipcfp_generate_event_proof
 * (IPCFP_WITNESS_BY_REFERENCE, IPCFP_SCAN_SKIP_TX_AMTS); the sharded flags give IPCFP_ERR_INVALID_ARG. A failure is the one B
 * reports: setup, message-AMT walk and pass-1 faults, then spec 0's pass-2 faults, spec 0's missing base-witness block, spec 1's
 * pass-2 faults, and so on. The offset arrays (n_specs + 1 entries each) belong to the caller. The result is an ordinary
 * ipcfp_event_result for ipcfp_event_result_free, ipcfp_event_result_to_json and ipcfp_verify_event_proofs. */
#define IPCFP_MAX_EVENT_SPECS 64
ipcfp_status ipcfp_generate_event_proof_multi(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* specs, uint32_t n_specs,
                                              uint32_t flags, uint64_t* spec_match_offsets, uint64_t* spec_proof_offsets,
                                              ipcfp_event_result** out);

/* Device-resident tipset descriptor: upload once, scan many specs against it (the reference calls
 * generate_event_proof once per EventProofSpec with the same tipsets, proofs/generator.rs:58-78). */
typedef struct ipcfp_tipset ipcfp_tipset;
ipcfp_status ipcfp_tipset_upload(ipcfp_store* s, const ipcfp_tipset_desc* t, ipcfp_tipset** out);
void ipcfp_tipset_free(ipcfp_tipset* t);
ipcfp_status ipcfp_generate_event_proof_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec, uint32_t flags,
                                                 ipcfp_event_result** out);
ipcfp_status ipcfp_generate_event_proof_shard_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec, uint64_t lo,
                                                       uint64_t hi, uint32_t world_size, uint32_t rank, uint32_t flags,
                                                       ipcfp_event_result** out);
/* ipcfp_generate_event_proof_multi against a device-resident tipset */
ipcfp_status ipcfp_generate_event_proof_multi_resident(ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* specs, uint32_t n_specs,
                                                       uint32_t flags, uint64_t* spec_match_offsets, uint64_t* spec_proof_offsets,
                                                       ipcfp_event_result** out);
/* The CUDA stream (cudaStream_t) all work of this store is issued on — for callers that time with
 * CUDA events or order their own device work after the engine's. */
void* ipcfp_store_stream(ipcfp_store* s);

/* read_storage_slot (src/proofs/storage/decode.rs:36-97), batched over k slot keys against one
 * contract_state root, with a RecordingBlockStore-equivalent witness. */
ipcfp_status ipcfp_read_storage_slots(ipcfp_store* s, const uint8_t contract_state_root[IPCFP_CID_LEN],
                                      const uint8_t* slots /* k*32 */, uint64_t k, ipcfp_slot_result** out);
void ipcfp_slot_result_free(ipcfp_slot_result* r);

/* generate_storage_proof (src/proofs/storage/generator.rs:29-67), batched over specs. */
ipcfp_status ipcfp_generate_storage_proofs(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_spec* specs,
                                           uint64_t n_specs, ipcfp_storage_result** out);
void ipcfp_storage_result_free(ipcfp_storage_result* r);

/* generate_proof_bundle (src/proofs/generator.rs:25-95). */
ipcfp_status ipcfp_generate_proof_bundle(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_storage_spec* sspecs,
                                         uint64_t n_sspecs, const ipcfp_event_spec* especs, uint64_t n_especs,
                                         ipcfp_bundle** out);
void ipcfp_bundle_free(ipcfp_bundle* b);

/* ------------------------------------------------------------------------------------------
 * Wire format (src/proofs/common/bundle.rs:10-45, src/proofs/events/bundle.rs:5-30, src/proofs/storage/bundle.rs:5-14): the JSON
 * `serde_json::to_string` gives for UnifiedProofBundle / EventProofBundle — struct field order, compact, CIDs as "bafy2bzace…"
 * strings, "0x" lower-case hex, base64 block data (ProofBlock.cid as the byte array cid 0.11's Serialize emits). t supplies the
 * fields every proof of the bundle shares (epochs, parent tipset CIDs, child block CID, parent state root). Host-side rendering:
 * no device is needed. *out is a NUL-terminated string of *out_len bytes, released with ipcfp_json_free.
 * ------------------------------------------------------------------------------------------ */
ipcfp_status ipcfp_bundle_to_json(const ipcfp_bundle* b, const ipcfp_tipset_desc* t, char** out, uint64_t* out_len);
ipcfp_status ipcfp_event_result_to_json(const ipcfp_event_result* r, const ipcfp_tipset_desc* t, char** out, uint64_t* out_len);
void ipcfp_json_free(char* p);

/* The way back (csrc/bundle_parse.cpp, host C++): what serde_json::from_str::<UnifiedProofBundle> / ::<EventProofBundle> reads, as
 * the PODs the batched verifiers below take and the flat block arrays ipcfp_store_create takes for the witness store. `tipset` holds
 * the fields every proof of the bundle shares (parent_epoch, child_epoch, n_parents, parent_cids, child_cid,
 * child_parent_state_root; the other members are NULL / 0); a bundle whose proofs disagree on them, CIDs that are not 38 bytes or
 * topics that are not 32 bytes are refused with IPCFP_ERR_UNSUPPORTED, malformed JSON / hex / base32 / base64 with
 * IPCFP_ERR_INVALID_ARG. Blocks are kept in the order given (16-byte aligned inside `witness.blob`); storage proofs come back with
 * found = 1, raw_len = 32 (the wire format carries the padded value only). No device is needed. */
typedef struct ipcfp_parsed_bundle {
    ipcfp_tipset_desc tipset;
    uint64_t n_storage_proofs;
    const ipcfp_storage_proof* storage_proofs;
    uint64_t n_event_proofs;
    const ipcfp_event_proof* event_proofs;
    const uint8_t* data_blob;          /* topics / data of the event proofs (topics_off / data_off index it) */
    uint64_t data_blob_size;
    ipcfp_witness witness;             /* Vec<ProofBlock> */
} ipcfp_parsed_bundle;
ipcfp_status ipcfp_bundle_from_json(const char* json, uint64_t len, ipcfp_parsed_bundle** out);
void ipcfp_parsed_bundle_free(ipcfp_parsed_bundle* b);

/* ------------------------------------------------------------------------------------------
 * Batched verifiers (src/proofs/events/verifier.rs:51-290, src/proofs/storage/verifier.rs:24-170): replay every proof against a
 * store that holds ONLY the witness blocks. Create that store with IPCFP_STORE_VERIFY_CIDS: this is the Blake2b-256 check of every
 * witness block the reference's load_witness_store leaves out (`put_keyed`, events/verifier.rs:79-89). results[i] = the reference's
 * Ok(bool) for proof i; an Err of the reference (missing witness block, decode failure, TxMeta mismatch) fails the call, index =
 * the first proof that meets it. Trust anchors (:124-144) are host-side policy closures and stay with the caller; `filter` (may
 * be NULL) plays check_event: the event must satisfy matches_log of that spec (events/generator.rs:38-40).
 * t: parent_cids / n_parents / epochs / child_cid (events), child_cid / child_parent_state_root (storage) — the fields every
 * proof of one bundle shares (EventProof.parent_tipset_cids …, StorageProof.parent_state_root).
 * ------------------------------------------------------------------------------------------ */
ipcfp_status ipcfp_verify_event_proofs(ipcfp_store* witness_store, const ipcfp_tipset_desc* t, const ipcfp_event_proof* proofs, uint64_t n_proofs,
                                       const uint8_t* data_blob, uint64_t data_blob_size, const ipcfp_event_spec* filter, uint8_t* results);
ipcfp_status ipcfp_verify_storage_proofs(ipcfp_store* witness_store, const ipcfp_tipset_desc* t, const ipcfp_storage_proof* proofs, uint64_t n_proofs,
                                         uint8_t* results);

/* ------------------------------------------------------------------------------------------
 * Multi-GPU (one process per GPU; the caller owns the communicator — torch.distributed / NCCL).
 * Receipts shard by index range; each rank scans its shard, then the per-shard witness CID sets
 * are all-gathered and merged (the BTreeSet union of src/proofs/common/witness.rs:24-40).
 * ------------------------------------------------------------------------------------------ */
/* In-library protocol (the reference's future-work "Parallel Generation", README.md:384; SURVEY Appendix C): one communicator
 * per process/GPU over NCCL (resolved with dlopen("libnccl.so.2") at init — the library itself links only cudart). Rank 0 makes
 * the id and hands the 128 bytes to the other ranks by any means (MPI, a file, torch.distributed …).
 * ipcfp_generate_event_proof_sharded = generate_event_proof (src/proofs/events/generator.rs:60-107) for ONE tipset whose
 * receipts are split by index range bounds[rank] .. bounds[rank+1] (bounds: world+1 ascending values, bounds[0] = 0,
 * bounds[world] = n_receipts); every rank's store holds the blocks its range needs (events blocks, receipts-AMT paths, its share
 * of the message AMTs, the shared top levels). Inside the call: all-to-all + all-reduce for the first-seen dedup of the
 * execution order (src/proofs/events/utils.rs:48-94), exec index → message CID fetch for the rank's proofs, and the union of the
 * per-shard witness CID sets (range-partitioned all-to-all + merge; see ipcfp_event_result.union_*). All ranks must make the call; they succeed or fail together and a
 * failure names the same (status, index) everywhere — the one the reference's sequential order meets first over all shards.
 * Errors: IPCFP_ERR_NCCL (library missing / communicator failure). */
#define IPCFP_COMM_ID_BYTES 128
typedef struct ipcfp_comm ipcfp_comm;
ipcfp_status ipcfp_comm_unique_id(uint8_t id[IPCFP_COMM_ID_BYTES]);
ipcfp_status ipcfp_comm_init(const uint8_t id[IPCFP_COMM_ID_BYTES], uint32_t world_size, uint32_t rank, int device, ipcfp_comm** out);
void ipcfp_comm_destroy(ipcfp_comm* c);
ipcfp_status ipcfp_generate_event_proof_sharded(ipcfp_comm* c, ipcfp_store* s, ipcfp_tipset* t, const ipcfp_event_spec* spec,
                                                const uint64_t* bounds /* world_size + 1 */, uint32_t flags, ipcfp_event_result** out);

/* Lower-level pieces (the caller owns the collectives — e.g. torch.distributed with the gloo backend on hosts without NCCL):
 * scan receipts [lo, hi) only. events_roots/has_events_root in t cover ALL n_receipts. */
ipcfp_status ipcfp_generate_event_proof_shard(ipcfp_store* s, const ipcfp_tipset_desc* t, const ipcfp_event_spec* spec,
                                              uint64_t lo, uint64_t hi, uint32_t world_size, uint32_t rank,
                                              uint32_t flags, ipcfp_event_result** out);
/* Cross-shard execution order (events/utils.rs:56-91, "first seen wins" over ALL message AMTs): a distributed
 * hash join whose collectives the caller runs between these device helpers. All pointers *_dev are device
 * memory; an "exec entry" is 48 bytes {record[40], global position u64}.
 *   1. pos0 = sum of shard_exec_count of lower ranks (all-gather); ipcfp_exec_bucketize routes every record of
 *      the rank's slice to owner = hash(cid) % world: send_dev = world segments of `cap` entries, counts[world].
 *      Inside a segment the entries are in increasing position order.
 *   2. all-to-all of counts and segments (segment r of the received buffer comes from rank r, so the buffer is
 *      ordered by global position per CID); ipcfp_exec_dedup returns the global positions that are NOT the first
 *      occurrence of their CID (any order).
 *   3. all-gather of the duplicate lists → sorted D on every rank: exec index i ↔ raw position p with
 *      p = i + |{d ∈ D : d ≤ p}|; n_exec = shard_raw_total − |D|.
 *   4. ipcfp_exec_fetch writes the records at the requested global positions this rank holds (others untouched). */
ipcfp_status ipcfp_exec_bucketize(int device, const void* seg_dev, uint64_t nseg, uint64_t pos0, uint32_t world, uint64_t cap,
                                  void* send_dev, uint64_t* counts /* host, world */);
ipcfp_status ipcfp_exec_dedup(int device, const void* recv_dev, const uint64_t* counts /* host, world */, uint32_t world, uint64_t cap,
                              uint64_t* dup_pos_dev, uint64_t cap_out, uint64_t* n_dup);
ipcfp_status ipcfp_exec_fetch(int device, const void* seg_dev, uint64_t nseg, uint64_t pos0, const uint64_t* req_pos_dev, uint64_t n_req,
                              void* out_dev /* n_req*40 */);
/* Device-resident copy of a result's sorted witness CIDs (n*38 bytes) for the collective. */
ipcfp_status ipcfp_witness_cids_to_device(const ipcfp_event_result* r, void* dev_ptr, uint64_t cap_cids, uint64_t* n);
/* Merge all-gathered CID lists on the device: gathered = world*cap*38 bytes, counts[world];
 * out_dev receives the sorted unique union (cap_out*38), *n_out its length. */
ipcfp_status ipcfp_merge_witness_cids(int device, const void* gathered_dev, const uint64_t* counts, uint32_t world,
                                      uint64_t cap, void* out_dev, uint64_t cap_out, uint64_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* IPCFP_H */
