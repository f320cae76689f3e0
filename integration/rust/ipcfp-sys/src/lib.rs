//! Raw bindings of `include/ipcfp.h` (what `bindgen` emits, written out by hand).
//! NOT BUILT IN THIS REPO: the build image has no Rust toolchain. Every item mirrors the C header one to one;
//! the reference-side shim (`GpuBlockstore`, `generate_event_proof_gpu`) is sketched in INTEGRATION.md §3.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const IPCFP_CID_LEN: usize = 38;
pub type ipcfp_status = i32;
pub const IPCFP_OK: ipcfp_status = 0;
pub const IPCFP_ERR_INVALID_ARG: ipcfp_status = -1;
pub const IPCFP_ERR_MISSING_BLOCK: ipcfp_status = -2;
pub const IPCFP_ERR_DECODE: ipcfp_status = -3;
pub const IPCFP_ERR_CID_MISMATCH: ipcfp_status = -4;
pub const IPCFP_ERR_MISSING_EXEC: ipcfp_status = -5;
pub const IPCFP_ERR_CUDA: ipcfp_status = -6;
pub const IPCFP_ERR_NCCL: ipcfp_status = -7;
pub const IPCFP_ERR_STATE_ROOT_MISMATCH: ipcfp_status = -8;
pub const IPCFP_ERR_ACTOR_NOT_FOUND: ipcfp_status = -9;
pub const IPCFP_ERR_NO_DEVICE: ipcfp_status = -10;
pub const IPCFP_ERR_UNSUPPORTED: ipcfp_status = -11;
pub const IPCFP_STORE_VERIFY_CIDS: u32 = 0x1;
pub const IPCFP_SCAN_SKIP_TX_AMTS: u32 = 0x1;
pub const IPCFP_SHARDED_UNION_TO_HOST: u32 = 0x2;
pub const IPCFP_SHARDED_UNION_FULL: u32 = 0x4;
pub const IPCFP_WITNESS_BY_REFERENCE: u32 = 0x8;
pub const IPCFP_COMM_ID_BYTES: usize = 128;
pub const IPCFP_MAX_EVENT_SPECS: u32 = 64;

#[repr(C)] pub struct ipcfp_store { _p: [u8; 0] }
#[repr(C)] pub struct ipcfp_tipset { _p: [u8; 0] }
#[repr(C)] pub struct ipcfp_comm { _p: [u8; 0] }

#[repr(C)]
pub struct ipcfp_tipset_desc {
    pub parent_epoch: i64,
    pub child_epoch: i64,
    pub n_parents: u32,
    pub parent_cids: *const u8,
    pub parent_txmeta_cids: *const u8,
    pub child_cid: *const u8,
    pub receipts_root: *const u8,
    pub child_parent_state_root: *const u8,
    pub n_receipts: u64,
    pub events_roots: *const u8,
    pub has_events_root: *const u8,
}
#[repr(C)]
pub struct ipcfp_event_spec { pub event_signature: *const c_char, pub topic_1: *const c_char, pub has_actor_id_filter: u8, pub actor_id_filter: u64 }
#[repr(C)]
pub struct ipcfp_storage_spec { pub actor_id: u64, pub slot: [u8; 32] }
#[repr(C)]
pub struct ipcfp_witness { pub n_blocks: u64, pub cids: *const u8, pub offsets: *const u64, pub lengths: *const u32, pub blob: *const u8, pub blob_size: u64 }
#[repr(C)]
pub struct ipcfp_event_proof {
    pub exec_index: u64, pub event_index: u64, pub emitter: u64, pub n_topics: u32, pub data_len: u32,
    pub data_off: u64, pub topics_off: u64, pub message_cid: [u8; IPCFP_CID_LEN], pub _pad: [u8; 2],
}
#[repr(C)]
pub struct ipcfp_event_result {
    pub n_matching: u64, pub matching_indices: *const u64, pub n_proofs: u64, pub proofs: *const ipcfp_event_proof,
    pub data_blob: *const u8, pub data_blob_size: u64, pub witness: ipcfp_witness, pub n_exec: u64,
    pub ms_total: f32, pub ms_pass1: f32, pub ms_pass2: f32, pub ms_txamt: f32, pub ms_witness: f32,
    pub pass1_bytes: u64, pub pass1_nodes: u64,
    pub shard_exec_dev: *const c_void, pub shard_exec_count: u64, pub shard_raw_total: u64,
    pub union_cids_dev: *const c_void, pub n_union_cids: u64, pub union_cids: *const u8, pub total_matching: u64, pub total_proofs: u64,
    pub ms_exchange: f32, pub ms_fetch: f32, pub ms_union: f32, pub _pad0: f32,
    pub union_part_first: u64, pub n_union_part: u64,
}
#[repr(C)]
pub struct ipcfp_storage_proof {
    pub actor_id: u64, pub actor_state_cid: [u8; IPCFP_CID_LEN], pub storage_root: [u8; IPCFP_CID_LEN],
    pub slot: [u8; 32], pub value: [u8; 32], pub found: u8, pub _pad: [u8; 3], pub raw_len: u32,
}
#[repr(C)]
pub struct ipcfp_storage_result {
    pub n_proofs: u64, pub proofs: *const ipcfp_storage_proof, pub witness: ipcfp_witness,
    pub spec_witness_offsets: *const u64, pub spec_witness_index: *const u32, pub ms_total: f32,
}
#[repr(C)]
pub struct ipcfp_slot_result { pub n: u64, pub found: *const u8, pub raw_len: *const u32, pub values: *const u8, pub witness: ipcfp_witness, pub ms_total: f32, pub ms_lookup: f32,
                                pub lookup_nodes: u64, pub lookup_bytes: u64 }
#[repr(C)]
pub struct ipcfp_parsed_bundle { pub tipset: ipcfp_tipset_desc, pub n_storage_proofs: u64, pub storage_proofs: *const ipcfp_storage_proof,
                                 pub n_event_proofs: u64, pub event_proofs: *const ipcfp_event_proof, pub data_blob: *const u8, pub data_blob_size: u64,
                                 pub witness: ipcfp_witness }
#[repr(C)]
pub struct ipcfp_bundle { pub storage: *mut ipcfp_storage_result, pub n_event_results: u64, pub events: *mut *mut ipcfp_event_result, pub witness: ipcfp_witness }

extern "C" {
    pub fn ipcfp_last_error() -> *const c_char;
    pub fn ipcfp_last_error_index() -> u64;
    pub fn ipcfp_version() -> *const c_char;
    pub fn ipcfp_kernel_launch_count() -> u64;
    pub fn ipcfp_host_alloc(bytes: usize, out: *mut *mut c_void) -> ipcfp_status;
    pub fn ipcfp_host_free(p: *mut c_void);

    pub fn ipcfp_store_create(cids: *const u8, offsets: *const u64, lengths: *const u32, blob: *const u8, blob_size: u64,
                              n_blocks: u64, device: c_int, flags: u32, out: *mut *mut ipcfp_store) -> ipcfp_status;
    pub fn ipcfp_store_destroy(s: *mut ipcfp_store);
    pub fn ipcfp_store_n_blocks(s: *const ipcfp_store) -> u64;
    pub fn ipcfp_store_get(s: *mut ipcfp_store, cid: *const u8, buf: *mut u8, cap: u32, len: *mut u32, found: *mut c_int) -> ipcfp_status;
    pub fn ipcfp_store_has(s: *mut ipcfp_store, cid: *const u8, found: *mut c_int) -> ipcfp_status;
    pub fn ipcfp_store_first_bad_block(s: *const ipcfp_store) -> u64;
    pub fn ipcfp_store_stream(s: *mut ipcfp_store) -> *mut c_void;

    pub fn ipcfp_blake2b256_batch(blob: *const u8, blob_size: u64, offsets: *const u64, lengths: *const u32, n: u64, device: c_int, out: *mut u8) -> ipcfp_status;
    pub fn ipcfp_keccak256_batch(blob: *const u8, blob_size: u64, offsets: *const u64, lengths: *const u32, n: u64, device: c_int, out: *mut u8) -> ipcfp_status;
    pub fn ipcfp_sha256_batch(blob: *const u8, blob_size: u64, offsets: *const u64, lengths: *const u32, n: u64, device: c_int, out: *mut u8) -> ipcfp_status;
    pub fn ipcfp_compute_mapping_slots(keys32: *const u8, slot_indices: *const u64, n: u64, device: c_int, out: *mut u8) -> ipcfp_status;

    pub fn ipcfp_generate_event_proof(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, spec: *const ipcfp_event_spec, flags: u32,
                                      out: *mut *mut ipcfp_event_result) -> ipcfp_status;
    pub fn ipcfp_event_result_free(r: *mut ipcfp_event_result);
    pub fn ipcfp_generate_event_proof_multi(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, specs: *const ipcfp_event_spec, n_specs: u32, flags: u32,
                                            spec_match_offsets: *mut u64, spec_proof_offsets: *mut u64,
                                            out: *mut *mut ipcfp_event_result) -> ipcfp_status;
    pub fn ipcfp_generate_event_proof_multi_resident(s: *mut ipcfp_store, t: *mut ipcfp_tipset, specs: *const ipcfp_event_spec, n_specs: u32, flags: u32,
                                                     spec_match_offsets: *mut u64, spec_proof_offsets: *mut u64,
                                                     out: *mut *mut ipcfp_event_result) -> ipcfp_status;
    pub fn ipcfp_tipset_upload(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, out: *mut *mut ipcfp_tipset) -> ipcfp_status;
    pub fn ipcfp_tipset_free(t: *mut ipcfp_tipset);
    pub fn ipcfp_generate_event_proof_resident(s: *mut ipcfp_store, t: *mut ipcfp_tipset, spec: *const ipcfp_event_spec, flags: u32,
                                               out: *mut *mut ipcfp_event_result) -> ipcfp_status;
    pub fn ipcfp_generate_event_proof_shard(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, spec: *const ipcfp_event_spec, lo: u64, hi: u64,
                                            world_size: u32, rank: u32, flags: u32, out: *mut *mut ipcfp_event_result) -> ipcfp_status;
    pub fn ipcfp_generate_event_proof_shard_resident(s: *mut ipcfp_store, t: *mut ipcfp_tipset, spec: *const ipcfp_event_spec, lo: u64, hi: u64,
                                                     world_size: u32, rank: u32, flags: u32, out: *mut *mut ipcfp_event_result) -> ipcfp_status;

    pub fn ipcfp_read_storage_slots(s: *mut ipcfp_store, contract_state_root: *const u8, slots: *const u8, k: u64, out: *mut *mut ipcfp_slot_result) -> ipcfp_status;
    pub fn ipcfp_slot_result_free(r: *mut ipcfp_slot_result);
    pub fn ipcfp_generate_storage_proofs(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, specs: *const ipcfp_storage_spec, n_specs: u64,
                                         out: *mut *mut ipcfp_storage_result) -> ipcfp_status;
    pub fn ipcfp_storage_result_free(r: *mut ipcfp_storage_result);
    pub fn ipcfp_generate_proof_bundle(s: *mut ipcfp_store, t: *const ipcfp_tipset_desc, sspecs: *const ipcfp_storage_spec, n_sspecs: u64,
                                       especs: *const ipcfp_event_spec, n_especs: u64, out: *mut *mut ipcfp_bundle) -> ipcfp_status;
    pub fn ipcfp_bundle_free(b: *mut ipcfp_bundle);

    pub fn ipcfp_bundle_to_json(b: *const ipcfp_bundle, t: *const ipcfp_tipset_desc, out: *mut *mut c_char, out_len: *mut u64) -> ipcfp_status;
    pub fn ipcfp_event_result_to_json(r: *const ipcfp_event_result, t: *const ipcfp_tipset_desc, out: *mut *mut c_char, out_len: *mut u64) -> ipcfp_status;
    pub fn ipcfp_json_free(p: *mut c_char);
    pub fn ipcfp_bundle_from_json(json: *const c_char, len: u64, out: *mut *mut ipcfp_parsed_bundle) -> ipcfp_status;
    pub fn ipcfp_parsed_bundle_free(b: *mut ipcfp_parsed_bundle);
    pub fn ipcfp_verify_event_proofs(witness_store: *mut ipcfp_store, t: *const ipcfp_tipset_desc, proofs: *const ipcfp_event_proof, n_proofs: u64,
                                     data_blob: *const u8, data_blob_size: u64, filter: *const ipcfp_event_spec, results: *mut u8) -> ipcfp_status;
    pub fn ipcfp_verify_storage_proofs(witness_store: *mut ipcfp_store, t: *const ipcfp_tipset_desc, proofs: *const ipcfp_storage_proof, n_proofs: u64,
                                       results: *mut u8) -> ipcfp_status;
    pub fn ipcfp_comm_unique_id(id: *mut u8) -> ipcfp_status;
    pub fn ipcfp_comm_init(id: *const u8, world_size: u32, rank: u32, device: c_int, out: *mut *mut ipcfp_comm) -> ipcfp_status;
    pub fn ipcfp_comm_destroy(c: *mut ipcfp_comm);
    pub fn ipcfp_generate_event_proof_sharded(c: *mut ipcfp_comm, s: *mut ipcfp_store, t: *mut ipcfp_tipset, spec: *const ipcfp_event_spec,
                                              bounds: *const u64, flags: u32, out: *mut *mut ipcfp_event_result) -> ipcfp_status;

    pub fn ipcfp_exec_bucketize(device: c_int, seg_dev: *const c_void, nseg: u64, pos0: u64, world: u32, cap: u64, send_dev: *mut c_void, counts: *mut u64) -> ipcfp_status;
    pub fn ipcfp_exec_dedup(device: c_int, recv_dev: *const c_void, counts: *const u64, world: u32, cap: u64, dup_pos_dev: *mut u64, cap_out: u64, n_dup: *mut u64) -> ipcfp_status;
    pub fn ipcfp_exec_fetch(device: c_int, seg_dev: *const c_void, nseg: u64, pos0: u64, req_pos_dev: *const u64, n_req: u64, out_dev: *mut c_void) -> ipcfp_status;
    pub fn ipcfp_witness_cids_to_device(r: *const ipcfp_event_result, dev_ptr: *mut c_void, cap_cids: u64, n: *mut u64) -> ipcfp_status;
    pub fn ipcfp_merge_witness_cids(device: c_int, gathered_dev: *const c_void, counts: *const u64, world: u32, cap: u64, out_dev: *mut c_void,
                                    cap_out: u64, n_out: *mut u64) -> ipcfp_status;
}
