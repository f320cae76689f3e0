"""Several event specs over the bench workload (1 M receipts x 8 events, store and tipset resident), three ways per spec count K:
  (a) ipcfp_generate_proof_bundle with the K specs and no storage specs (the existing way to serve a bundle's event specs),
  (b) K x ipcfp_generate_event_proof_resident,
  (c) ipcfp_generate_event_proof_multi_resident (one scan for all K).
The arms alternate within each repetition. Per arm: wall-clock ms per call (the calls end in a host synchronisation), device ms
(CUDA events of the calls: ms_total, summed over the K calls of (a) and (b)), pass-1 kernel ms, kernel launches per call. `parity`:
(c) equals (a) byte for byte under the contract of ipcfp_generate_event_proof_multi.

Spec mix: spec 0 is the workload's own target (actor filtered, ~0.1 % of receipts); of the others every fourth is high-rate
(OtherJ / calib-subnet-M, no actor filter, ~6 %) and the rest low-rate (the same with an actor filter, ~0.4 %).

    python tools/bench_multi.py [--reps 5] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from ipc_filecoin_proofs_b200 import _abi as A  # noqa: E402
from ipc_filecoin_proofs_b200 import api  # noqa: E402


def spec_mix(ts, K):
    specs = [A.make_event_spec(ts.event_signature, ts.topic1, ts.actor_filter)]
    for k in range(1, K):
        sig = f"Other{1 + k % 7}(bytes32,uint256)"
        subnet = f"calib-subnet-{(3 * k) % 16}"
        specs.append(A.make_event_spec(sig, subnet, None if k % 4 == 1 else 1000 + (k * 7) % 16))
    return specs


def records(ptr, n):
    dt = np.dtype([("exec_index", "<u8"), ("event_index", "<u8"), ("emitter", "<u8"), ("n_topics", "<u4"), ("data_len", "<u4"),
                   ("data_off", "<u8"), ("topics_off", "<u8"), ("message_cid", "u1", 38), ("_pad", "u1", 2)])
    return np.frombuffer(A._arr(C.cast(ptr, C.c_void_p).value, n * dt.itemsize, np.uint8).tobytes(), dtype=dt) if n else np.zeros(0, dt)


def witness_arrays(w):
    n = int(w.n_blocks)
    cids = A._arr(w.cids, 38 * n, np.uint8).copy()
    offs, lens = A._arr(w.offsets, n, np.uint64), A._arr(w.lengths, n, np.uint32)
    blob = A._arr(w.blob, int(w.blob_size), np.uint8)
    data = b"".join(blob[int(o):int(o) + int(l)].tobytes() for o, l in zip(offs, lens))
    return cids, lens.copy(), data


def parity(fused, mo, po, bundle):
    """fused (ipcfp_event_result) + offsets == bundle (ipcfp_bundle) under the multi call's contract."""
    r, b = fused, bundle
    K = int(b.n_event_results)
    mi = A._arr(r.matching_indices, int(r.n_matching), np.uint64)
    recs = records(r.proofs, int(r.n_proofs))
    blob = A._arr(r.data_blob, int(r.data_blob_size), np.uint8)
    base = 0
    for k in range(K):
        e = b.events[k].contents
        if not np.array_equal(mi[int(mo[k]):int(mo[k + 1])], A._arr(e.matching_indices, int(e.n_matching), np.uint64)):
            return False
        er = records(e.proofs, int(e.n_proofs)).copy()
        er["topics_off"] += base
        er["data_off"] += base
        if recs[int(po[k]):int(po[k + 1])].tobytes() != er.tobytes():
            return False
        eb = A._arr(e.data_blob, int(e.data_blob_size), np.uint8)
        if not np.array_equal(blob[base:base + len(eb)], eb):
            return False
        base += len(eb)
    if base != len(blob) or r.n_exec != b.events[0].contents.n_exec:
        return False
    wa, wb = witness_arrays(r.witness), witness_arrays(b.witness)
    return all(np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(wa, wb))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ks", default="1,2,4,8,16,64")
    ap.add_argument("--receipts", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import synth
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    emit({"gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"})
    ts = synth.Tipset(synth.config_params(4, n_receipts=args.receipts))
    L = api.lib()
    d, keep = A.make_tipset_desc(ts)
    store = api.BlockStore.from_tipset(ts)
    tip = store.upload_tipset(ts)
    emit({"workload": f"{ts.n_blocks} blocks, {args.receipts} receipts x 8 events"})

    def arm_bundle(specs):
        arr = (A.EventSpec * len(specs))(*specs)
        out = C.POINTER(A.BundleC)()
        assert L.ipcfp_generate_proof_bundle(store._h, C.byref(d), None, 0, arr, len(specs), C.byref(out)) == 0, L.ipcfp_last_error()
        b = out.contents
        dev = sum(b.events[k].contents.ms_total for k in range(len(specs)))
        p1 = sum(b.events[k].contents.ms_pass1 for k in range(len(specs)))
        return out, dev, p1, lambda: L.ipcfp_bundle_free(out)

    def arm_singles(specs):
        dev = p1 = 0.0
        for s in specs:
            out = C.POINTER(A.EventResultC)()
            assert L.ipcfp_generate_event_proof_resident(store._h, tip._h, C.byref(s), 0, C.byref(out)) == 0, L.ipcfp_last_error()
            dev += out.contents.ms_total
            p1 += out.contents.ms_pass1
            L.ipcfp_event_result_free(out)
        return None, dev, p1, lambda: None

    def arm_fused(specs, keep_offsets=None):
        arr = (A.EventSpec * len(specs))(*specs)
        mo, po = np.zeros(len(specs) + 1, np.uint64), np.zeros(len(specs) + 1, np.uint64)
        out = C.POINTER(A.EventResultC)()
        assert L.ipcfp_generate_event_proof_multi_resident(store._h, tip._h, arr, len(specs), 0, mo.ctypes.data, po.ctypes.data,
                                                            C.byref(out)) == 0, L.ipcfp_last_error()
        if keep_offsets is not None:
            keep_offsets.extend([mo, po])
        return out, out.contents.ms_total, out.contents.ms_pass1, lambda: L.ipcfp_event_result_free(out)

    arms = {"bundle": arm_bundle, "singles": arm_singles, "fused": arm_fused}
    for K in [int(k) for k in args.ks.split(",")]:
        specs = spec_mix(ts, K)
        # warm-up of every arm, then the parity check of (c) against (a)
        for f in arms.values():
            f(specs)[3]()
        offs = []
        fo, _, _, ffree = arm_fused(specs, offs)
        bo, _, _, bfree = arm_bundle(specs)
        ok = parity(fo.contents, offs[0], offs[1], bo.contents)
        n_match = [int(offs[0][k + 1] - offs[0][k]) for k in range(K)]
        ffree()
        bfree()
        res = {name: {"wall": [], "dev": [], "pass1": [], "launches": 0} for name in arms}
        for _ in range(args.reps):
            for name, f in arms.items():
                n0 = api.kernel_launch_count()
                t0 = time.perf_counter()
                _, dev, p1, free = f(specs)
                t1 = time.perf_counter()
                res[name]["launches"] = api.kernel_launch_count() - n0
                free()
                res[name]["wall"].append((t1 - t0) * 1e3)
                res[name]["dev"].append(dev)
                res[name]["pass1"].append(p1)
        line = {"K": K, "parity": bool(ok), "receipts_per_spec": n_match}
        for name, v in res.items():
            line[name] = {"wall_ms": round(float(np.median(v["wall"])), 3), "device_ms": round(float(np.median(v["dev"])), 3),
                          "pass1_ms": round(float(np.median(v["pass1"])), 3), "launches": v["launches"]}
        line["fused_speedup_vs_bundle"] = round(line["bundle"]["wall_ms"] / line["fused"]["wall_ms"], 2)
        line["fused_vs_singles"] = round(line["fused"]["wall_ms"] / line["singles"]["wall_ms"], 3)
        emit(line)
    tip.close()
    store.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
