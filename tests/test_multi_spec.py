"""ipcfp_generate_event_proof_multi: several event specs in one scan of the tipset, against the oracle's and the engine's
generate_proof_bundle (no storage specs) — per-spec matching receipts and proofs, one union witness, the same first failure."""
import ctypes as C

import numpy as np
import pytest

from ipc_filecoin_proofs_b200 import _abi as A
from tests.util import EditedTipset, ShuffledTipset, assert_witness_equal, spec_of

pytestmark = pytest.mark.gpu

SHAPES = [
    dict(n_receipts=300, events_per_receipt=40, match_ppm=100000),
    dict(n_receipts=500, events_per_receipt=3, null_root_permille=200, match_ppm=200000),
    dict(n_receipts=257, events_per_receipt=8, bw3_permille=1000, match_ppm=50000, has_actor_filter=0),
    dict(n_receipts=1000, events_per_receipt=8, case_a_permille=500, malformed_permille=100, match_ppm=30000),
    dict(n_receipts=1, events_per_receipt=1, match_ppm=1000000, dup_msgs=0, n_parents=1),
    dict(n_receipts=9, events_per_receipt=8, match_ppm=0, n_parents=3, dup_msgs=2),
    dict(n_receipts=700, events_per_receipt=300, match_ppm=20000, n_parents=1),
]


def _sig(j):
    return "NewTopDownMessage(bytes32,uint256)" if j == 0 else f"Other{j}(bytes32,uint256)"


def _topic(ts, j):
    # configs with same_topic1 carry calib-subnet-1 in every event: vary the signature and the actor filter there instead
    return ts.topic1 if ts.params.same_topic1 else f"calib-subnet-{j}"


def spec_sets(ts):
    tgt = spec_of(ts)
    plain = A.make_event_spec(ts.event_signature, ts.topic1, None)
    with_actor = A.make_event_spec(ts.event_signature, ts.topic1, 1003)
    other = A.make_event_spec(_sig(3), _topic(ts, 5), None)
    other_actor = A.make_event_spec(_sig(5), _topic(ts, 7), 1002)
    nothing = A.make_event_spec("Nothing(bytes32)", "no-such-subnet", None)
    many = [A.make_event_spec(_sig(j % 8), _topic(ts, (j * 5) % 16), (1000 + j % 16) if j % 3 == 0 else None) for j in range(62)]
    return {
        "target": [tgt],
        "target_twice": [tgt, tgt],
        "actor_filter": [plain, with_actor, tgt],
        "disjoint": [other, tgt, other_actor],
        "matches_nothing": [nothing, tgt, nothing],
        "k64": many + [tgt, plain],
    }


def _bundle(make_store, ts, specs):
    try:
        return ("ok", make_store().generate_proof_bundle(ts, [], specs))
    except A.IpcfpError as e:
        return ("err", e.status, e.index)


def _multi(api, ts, specs, flags=0, store=None):
    try:
        return ("ok", (store or api.BlockStore.from_tipset(ts)).generate_event_proof_multi(ts, specs, flags))
    except A.IpcfpError as e:
        return ("err", e.status, e.index)


def assert_multi_equals_bundle(m, b):
    """m: MultiEventResult, b: BundlePy of the same specs (the contract of ipcfp_generate_event_proof_multi)."""
    r = m.result
    K = len(b.events)
    assert len(m.match_offsets) == K + 1 and len(m.proof_offsets) == K + 1
    blob_base = 0
    for k, e in enumerate(b.events):
        mi, pr = m.spec(k)
        assert mi.tolist() == e.matching.tolist(), k
        assert [p.key() for p in pr] == [p.key() for p in e.proofs], k
        assert np.array_equal(r.data_blob[blob_base:blob_base + len(e.data_blob)], e.data_blob), k
        blob_base += len(e.data_blob)
    assert blob_base == len(r.data_blob)
    assert int(m.match_offsets[-1]) == len(r.matching) and int(m.proof_offsets[-1]) == len(r.proofs)
    assert r.n_exec == b.events[0].n_exec
    assert_witness_equal(r.witness, b.witness)


def _offsets_of(m, b):
    """(topics_off, data_off) of every proof of m, and the same of the bundle's proofs shifted by their spec's blob base."""
    got = [(int(x["topics_off"]), int(x["data_off"])) for x in _records(m.result)]
    exp, base = [], 0
    for e in b.events:
        exp += [(int(x["topics_off"]) + base, int(x["data_off"]) + base) for x in _records(e)]
        base += len(e.data_blob)
    return got, exp


def _records(res):
    dt = np.dtype([("exec_index", "<u8"), ("event_index", "<u8"), ("emitter", "<u8"), ("n_topics", "<u4"), ("data_len", "<u4"),
                   ("data_off", "<u8"), ("topics_off", "<u8"), ("message_cid", "u1", 38), ("_pad", "u1", 2)])
    assert dt.itemsize == C.sizeof(A.EventProofC)
    return np.frombuffer(res.raw_proofs.tobytes(), dtype=dt)


def check(api, oracle_mod, ts, specs):
    o = _bundle(lambda: oracle_mod.Store.from_tipset(ts), ts, specs)
    e = _bundle(lambda: api.BlockStore.from_tipset(ts), ts, specs)
    m = _multi(api, ts, specs)
    assert o[0] == e[0] == m[0], (o[:3], e[:3], m[:3])
    if o[0] != "ok":
        assert o[1:] == e[1:] == m[1:], (o, e, m)
        return None
    assert_multi_equals_bundle(m[1], o[1])
    assert_multi_equals_bundle(m[1], e[1])
    got, exp = _offsets_of(m[1], o[1])
    assert got == exp
    return m[1]


@pytest.mark.parametrize("cfg", [1, 2])
@pytest.mark.parametrize("which", ["target", "target_twice", "actor_filter", "disjoint", "matches_nothing", "k64"])
def test_multi_parity_configs(api, oracle_mod, synth_mod, cfg, which):
    ts = synth_mod.Tipset(synth_mod.config_params(cfg))
    specs = spec_sets(ts)[which]
    m = check(api, oracle_mod, ts, specs)
    if which == "matches_nothing":
        assert m.spec(0)[0].size == 0 and m.spec(2)[0].size == 0 and m.spec(1)[0].size > 0
    if which == "target_twice":
        assert m.spec(0)[0].tolist() == m.spec(1)[0].tolist() and len(m.spec(1)[1]) > 0
    # the resident variant gives the same result
    store = api.BlockStore.from_tipset(ts)
    tip = store.upload_tipset(ts)
    r = store.generate_event_proof_multi_resident(tip, specs)
    tip.close()
    assert r.result.matching.tolist() == m.result.matching.tolist() and np.array_equal(r.match_offsets, m.match_offsets)
    assert [p.key() for p in r.result.proofs] == [p.key() for p in m.result.proofs] and np.array_equal(r.proof_offsets, m.proof_offsets)
    assert np.array_equal(r.result.data_blob, m.result.data_blob) and np.array_equal(r.result.raw_proofs, m.result.raw_proofs)
    assert_witness_equal(r.result.witness, m.result.witness)


@pytest.mark.parametrize("kw", SHAPES)
def test_multi_parity_shapes(api, oracle_mod, synth_mod, kw):
    ts = synth_mod.Tipset(synth_mod.default_params(seed=99, **kw))
    sets = spec_sets(ts)
    for which in ("disjoint", "actor_filter", "k64"):
        check(api, oracle_mod, ts, sets[which])


def test_multi_parity_shuffled_misaligned(api, oracle_mod, ts2):
    sh = ShuffledTipset(ts2, seed=3, misalign=True)
    specs = spec_sets(ts2)["disjoint"] + [spec_of(ts2)]
    exp = oracle_mod.Store.from_tipset(ts2).generate_proof_bundle(ts2, [], specs)
    got = api.BlockStore.from_tipset(sh, verify_cids=True).generate_event_proof_multi(sh, specs)
    assert_multi_equals_bundle(got, exp)


@pytest.mark.parametrize("n_decoys", [0, 4])
def test_multi_both_pass2_shapes(api, oracle_mod, synth_mod, n_decoys):
    """Above 16 384 matching receipts pass 2 runs one receipt per thread, below one per warp: decoy specs of ~6 % each on
    300 k receipts push the union of the matches over the line."""
    ts = synth_mod.Tipset(synth_mod.default_params(seed=5, n_receipts=300_000, events_per_receipt=8, match_ppm=2000))
    decoys = [A.make_event_spec(_sig(j + 1), f"calib-subnet-{j + 2}", None) for j in range(n_decoys)]
    specs = [spec_of(ts)] + decoys
    m = check(api, oracle_mod, ts, specs)
    union = len(np.unique(m.result.matching))
    assert (union > 16384) == (n_decoys > 0), union


def test_multi_flags(api, oracle_mod, ts2):
    specs = spec_sets(ts2)["disjoint"]
    store = api.BlockStore.from_tipset(ts2)
    full = store.generate_event_proof_multi(ts2, specs)
    # witness by reference: the same CIDs and lengths, offsets into the blob the store was created from
    ref = store.generate_event_proof_multi(ts2, specs, A.WITNESS_BY_REFERENCE)
    assert np.array_equal(ref.result.witness.cids, full.result.witness.cids)
    assert np.array_equal(ref.result.witness.lengths, full.result.witness.lengths)
    assert ref.result.witness.blob.size == 0
    blocks = [bytes(ts2.blob[int(o):int(o) + int(n)]) for o, n in zip(ref.result.witness.offsets, ref.result.witness.lengths)]
    assert blocks == full.result.witness.blocks()
    assert [p.key() for p in ref.result.proofs] == [p.key() for p in full.result.proofs]
    # skip the message AMTs: per spec the single skip-flag call, the witness their union
    skip = store.generate_event_proof_multi(ts2, specs, A.SCAN_SKIP_TX_AMTS)
    singles = [store.generate_event_proof(ts2, s, A.SCAN_SKIP_TX_AMTS) for s in specs]
    cids = set()
    for k, s in enumerate(singles):
        mi, pr = skip.spec(k)
        assert mi.tolist() == s.matching.tolist() and [p.key() for p in pr] == [p.key() for p in s.proofs]
        cids |= {bytes(c) for c in s.witness.cids}
        assert s.n_exec == skip.result.n_exec
    assert {bytes(c) for c in skip.result.witness.cids} == cids and len(cids) == skip.result.witness.n_blocks
    # sharded flags and bad arguments are rejected
    for bad in (lambda: store.generate_event_proof_multi(ts2, specs, 0x2), lambda: store.generate_event_proof_multi(ts2, specs, 0x4),
                lambda: store.generate_event_proof_multi(ts2, []), lambda: store.generate_event_proof_multi(ts2, [specs[0]] * 65)):
        with pytest.raises(A.IpcfpError) as ei:
            bad()
        assert ei.value.status == A.ERR_INVALID_ARG
    d, keep = A.make_tipset_desc(ts2)
    arr = (A.EventSpec * 1)(specs[0])
    off = np.zeros(2, dtype=np.uint64)
    out = C.POINTER(A.EventResultC)()
    L = api.lib()
    assert L.ipcfp_generate_event_proof_multi(store._h, C.byref(d), arr, 1, 0, None, off.ctypes.data, C.byref(out)) == A.ERR_INVALID_ARG
    assert L.ipcfp_generate_event_proof_multi(store._h, C.byref(d), None, 1, 0, off.ctypes.data, off.ctypes.data, C.byref(out)) == A.ERR_INVALID_ARG


def _error_cases(ts1):
    import cbor2
    from tests.test_oracle_cpu import _patched
    d = ts1.as_dict()
    cases = []
    has = ts1.has_events_root.copy()
    has[::3] = 0
    cases.append(EditedTipset(ts1, has_events_root=has))

    def without(t, cid):
        keep = [i for i in range(t.n_blocks) if bytes(t.cids[i]) != bytes(cid)]
        return EditedTipset(t, cids=t.cids[keep], offsets=t.offsets[keep], lengths=t.lengths[keep], n_blocks=len(keep))
    cases.append(without(ts1, ts1.events_roots[5]))
    rr = cbor2.loads(d[bytes(ts1.receipts_root)])
    cases.append(without(ts1, rr[2][1][1].value[1:]))
    tm = cbor2.loads(d[bytes(ts1.parent_txmeta_cids[0])])
    bls_root = cbor2.loads(d[tm[0].value[1:]])
    cases.append(without(ts1, bls_root[2][1][0].value[1:]))
    cases.append(without(ts1, ts1.parent_txmeta_cids[1]))
    cases.append(without(ts1, ts1.parent_cids[0]))
    cases.append(without(ts1, ts1.receipts_root))
    ev = d[bytes(ts1.events_roots[9])]
    for bad in (ev + b"\x00", ev[:-1], ev[:1] + b"\x06" + ev[2:], ev[:5] + b"\x45\xff\x00\x00\x00\x00" + ev[10:], b"\xa0", b"",
                ev.replace(b"\x62t1", b"\x62t\xff", 1), ev.replace(b"\x18\x55\x58\x20", b"\x18\x17\x58\x20", 1),
                ev.replace(b"\x19\x03", b"\x1a\x00\x00\x03", 1)):
        cases.append(_patched(ts1, ts1.events_roots[9], bad))
    leaf_cid = rr[2][1][0].value[1:]
    leaf = d[leaf_cid]
    cases.append(_patched(ts1, leaf_cid, leaf[:-1]))
    cases.append(_patched(ts1, leaf_cid, leaf.replace(b"\x84\x00\x40", b"\x84\x20\x40", 1)))
    cases.append(_patched(ts1, ts1.parent_txmeta_cids[0], cbor2.dumps([tm[0]])))
    short = EditedTipset(ts1, parent_cids=ts1.parent_cids[:1], parent_txmeta_cids=ts1.parent_txmeta_cids[:1], n_parents=1)
    cases.append(short)
    cases.append(without(short, ts1.parent_cids[0]))   # exec.get faults together with a missing base-witness block
    return cases


def test_multi_error_parity(api, oracle_mod, ts1):
    """The fault kinds of test_error_parity, each under spec sets where the first fault is reached through different specs: only
    through spec 1's matches, through specs 0 and 2, with a missing base-witness block that ranks between spec 0's and spec 1's
    pass-2 faults. ts1 carries calib-subnet-1 in every event, so the specs differ by signature and actor filter."""
    t1 = ts1.topic1
    s = [A.make_event_spec(_sig(j), t1, None) for j in range(8)]
    sets = [
        [spec_of(ts1), s[3]],
        [A.make_event_spec("Nothing(bytes32)", t1, None), s[2]],            # spec 0 matches nothing: every pass-2 fault is spec 1's
        [s[4], s[1], s[4]],                                                 # specs 0 and 2 identical
        [A.make_event_spec(_sig(0), t1, 1001), s[5], s[0], s[6]],
    ]
    seen = {"ok": 0, "err": 0, "spec1": 0}
    for k, ts in enumerate(_error_cases(ts1)):
        for specs in sets:
            o = _bundle(lambda: oracle_mod.Store.from_tipset(ts), ts, specs)
            e = _bundle(lambda: api.BlockStore.from_tipset(ts), ts, specs)
            m = _multi(api, ts, specs)
            assert o[0] == e[0] == m[0], (k, o[:3], e[:3], m[:3])
            if o[0] == "ok":
                seen["ok"] += 1
                assert_multi_equals_bundle(m[1], o[1])
            else:
                seen["err"] += 1
                assert o[1:] == e[1:] == m[1:], (k, o, e, m)
                # a fault met in the reference's spec-1 call: the single call of spec 0 alone succeeds
                if _bundle(lambda: oracle_mod.Store.from_tipset(ts), ts, specs[:1])[0] == "ok":
                    seen["spec1"] += 1
    assert seen["ok"] > 0 and seen["err"] > 40 and seen["spec1"] > 0, seen


def test_multi_closed_loop(api, oracle_mod, ts2):
    specs = spec_sets(ts2)["disjoint"] + [spec_of(ts2)]
    store = api.BlockStore.from_tipset(ts2)
    m = store.generate_event_proof_multi(ts2, specs)
    assert all(api.verify_event_proofs(m.result.witness, ts2, m.result))
    assert all(oracle_mod.verify_event_proofs(m.result.witness, ts2, m.result))
    sz = C.sizeof(A.EventProofC)

    class Part:
        pass
    for k, sp in enumerate(specs):
        a, b = int(m.proof_offsets[k]), int(m.proof_offsets[k + 1])
        p = Part()
        p.proofs = m.result.proofs[a:b]
        p.raw_proofs = m.result.raw_proofs[a * sz:b * sz]
        p.data_blob = m.result.data_blob
        ok = api.verify_event_proofs(m.result.witness, ts2, p, sp)
        assert len(ok) == b - a and all(ok), k
    # the JSON EventProofBundle of the fused result parses back to the same proofs and blocks
    d, keep = A.make_tipset_desc(ts2)
    arr = (A.EventSpec * len(specs))(*specs)
    mo, po = np.zeros(len(specs) + 1, dtype=np.uint64), np.zeros(len(specs) + 1, dtype=np.uint64)
    out = C.POINTER(A.EventResultC)()
    L = api.lib()
    assert L.ipcfp_generate_event_proof_multi(store._h, C.byref(d), arr, len(specs), 0, mo.ctypes.data, po.ctypes.data, C.byref(out)) == 0
    try:
        pb = api.ParsedBundle(api.event_result_to_json(out, ts2))
        raw, blob = pb.event_proofs_raw
        rec = np.frombuffer(raw.tobytes(), dtype=_records(m.result).dtype)
        mine = _records(m.result)
        assert len(rec) == len(mine)
        for x, y in zip(rec, mine):
            assert x["exec_index"] == y["exec_index"] and x["event_index"] == y["event_index"] and x["emitter"] == y["emitter"]
            assert bytes(x["message_cid"]) == bytes(y["message_cid"])
            assert bytes(blob[x["topics_off"]:x["topics_off"] + 32 * x["n_topics"]]) == \
                bytes(m.result.data_blob[y["topics_off"]:y["topics_off"] + 32 * y["n_topics"]])
            assert bytes(blob[x["data_off"]:x["data_off"] + x["data_len"]]) == bytes(m.result.data_blob[y["data_off"]:y["data_off"] + y["data_len"]])
        assert_witness_equal(pb.witness, m.result.witness)
        pb.close()
    finally:
        L.ipcfp_event_result_free(out)


def test_multi_launch_count_does_not_depend_on_k(api, ts2):
    store = api.BlockStore.from_tipset(ts2)
    sets = spec_sets(ts2)
    store.generate_event_proof_multi(ts2, sets["target"])     # warm-up
    counts = {}
    for name, specs in (("k1", sets["target"]), ("k8", (sets["disjoint"] + sets["actor_filter"] + sets["target_twice"])[:8]), ("k64", sets["k64"])):
        n0 = api.kernel_launch_count()
        store.generate_event_proof_multi(ts2, specs)
        counts[name] = api.kernel_launch_count() - n0
    n0 = api.kernel_launch_count()
    store.generate_event_proof(ts2, spec_of(ts2))
    single = api.kernel_launch_count() - n0
    assert counts["k1"] == counts["k8"] == counts["k64"], counts
    # the pair compaction and the pair scans take two launches each whatever their size; the single call's per-receipt scans take one
    # each at this size and two at 1 M receipts: 9 more launches than the single call here, 7 more (48 vs 41) at 1 M receipts
    assert counts["k1"] <= single + 9, (counts, single)
