"""The ctypes mirror (ipc_filecoin_proofs_b200/_abi.py) must have exactly the C layout of include/ipcfp.h,
and the Rust binding source must declare every exported function."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from ipc_filecoin_proofs_b200 import _abi as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STRUCTS = {
    "ipcfp_tipset_desc": A.TipsetDesc, "ipcfp_event_spec": A.EventSpec, "ipcfp_storage_spec": A.StorageSpec, "ipcfp_witness": A.Witness,
    "ipcfp_event_proof": A.EventProofC, "ipcfp_event_result": A.EventResultC, "ipcfp_storage_proof": A.StorageProofC,
    "ipcfp_storage_result": A.StorageResultC, "ipcfp_slot_result": A.SlotResultC, "ipcfp_bundle": A.BundleC,
    "ipcfp_parsed_bundle": A.ParsedBundleC,
}


def test_ctypes_layout_matches_c_header():
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ipcfp.h"', "int main(void) {"]
    for cname, st in STRUCTS.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in st._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["return 0; }"]
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "layout.c")
        exe = os.path.join(td, "layout")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, src])
        out = subprocess.check_output([exe], text=True)
    got = dict(l.split() for l in out.strip().splitlines())
    for cname, st in STRUCTS.items():
        assert int(got[cname]) == C.sizeof(st), cname
        for fname, _ in st._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(st, fname).offset, f"{cname}.{fname}"


def test_rust_sys_source_declares_every_export():
    hdr = open(os.path.join(ROOT, "include", "ipcfp.h")).read()
    declared = set(re.findall(r"\b(ipcfp_[a-z0-9_]+)\s*\(", hdr)) - {"ipcfp_store", "ipcfp_tipset"}
    rs = open(os.path.join(ROOT, "integration", "rust", "ipcfp-sys", "src", "lib.rs")).read()
    rust = set(re.findall(r"pub fn (ipcfp_[a-z0-9_]+)\s*\(", rs))
    assert declared == rust, (declared - rust, rust - declared)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` prints exactly one JSON line with the contract's keys (tiny workload)."""
    import json
    import sys
    env = dict(os.environ, IPCFP_BENCH_RECEIPTS="3000")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                                  env=env, text=True, stderr=subprocess.DEVNULL)
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "receipts/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0


def _bench_dump(out_dir, *argv):
    """bench.py on a 3000-receipt tipset with `--dump-outputs out_dir` → (its JSON line, {name: array} of what it wrote)."""
    import json
    import sys
    env = dict(os.environ, IPCFP_BENCH_RECEIPTS="3000")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), *argv, "--dump-outputs", str(out_dir)], env=env, text=True,
                                  stderr=subprocess.DEVNULL)
    return json.loads(out), {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_bench_dump_outputs_reference_arm(tmp_path, synth_mod, oracle_mod):
    """`bench.py --dump-outputs DIR` writes the last timed step's result as float32 / float64 arrays; the same arguments give the same
    inputs, so two runs (of different --steps) write the same arrays, and they are the oracle's result on the benchmark's tipset."""
    (la, a), (lb, b) = [_bench_dump(tmp_path / str(k), "--impl", "reference", "--steps", str(k), "--warmup", "0") for k in (1, 2)]
    assert (la["steps"], lb["steps"]) == (1, 2)
    assert sorted(a) == sorted(b) == ["counts", "matching", "proof_fields", "proof_message_cids", "proof_payload", "witness_bytes",
                                      "witness_cids", "witness_lengths"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    ts = synth_mod.Tipset(synth_mod.config_params(4, n_receipts=3000))
    exp = oracle_mod.Store.from_tipset(ts).generate_event_proof(ts, A.make_event_spec(ts.event_signature, ts.topic1, ts.actor_filter))
    blocks = b"".join(exp.witness.blocks())
    assert a["counts"].tolist() == [len(exp.matching), len(exp.proofs), exp.n_exec, exp.witness.n_blocks, len(blocks)]
    assert len(exp.proofs) > 0 and exp.witness.n_blocks > 0
    assert np.array_equal(a["matching"], exp.matching) and np.array_equal(a["witness_cids"], exp.witness.cids)
    assert np.array_equal(a["witness_lengths"], exp.witness.lengths) and np.array_equal(a["witness_bytes"], np.frombuffer(blocks, np.uint8))
    assert a["proof_fields"][:, 0].tolist() == [p.exec_index for p in exp.proofs]
    assert np.array_equal(a["proof_message_cids"], np.array([list(p.message_cid) for p in exp.proofs]))
    assert np.array_equal(a["proof_payload"], np.frombuffer(b"".join(b"".join(p.topics) + p.data for p in exp.proofs), np.uint8))


@pytest.mark.gpu
def test_bench_dump_outputs_engine_equals_reference_arm(tmp_path):
    """The engine arm's dump equals the reference arm's array for array on the same inputs, and --steps sets the number of timed
    steps: the kernel launches counted over the timed region grow with it."""
    _, ref = _bench_dump(tmp_path / "ref", "--impl", "reference", "--steps", "1", "--warmup", "0")
    (l2, g2), (l3, g3) = [_bench_dump(tmp_path / str(k), "--steps", str(k), "--warmup", "1", "--no-storage", "--no-cpu-baseline") for k in (2, 3)]
    for got in (g2, g3):
        assert sorted(got) == sorted(ref)
        for k in ref:
            assert np.array_equal(got[k], ref[k]), k
    assert (l2["steps"], l3["steps"]) == (2, 3)
    assert l3["gpu_launches"] > l2["gpu_launches"] > 0


def test_rust_shim_uses_only_declared_bindings():
    """integration/rust/gpu.rs cannot be compiled here (no Rust toolchain); at least every `sys::` item it names must exist in the -sys
    crate and every call must pass as many arguments as the declaration takes."""
    sys_rs = open(os.path.join(ROOT, "integration", "rust", "ipcfp-sys", "src", "lib.rs")).read()
    shim = open(os.path.join(ROOT, "integration", "rust", "gpu.rs")).read()
    fns = {m.group(1): m.group(2) for m in re.finditer(r"pub fn (ipcfp_[a-z0-9_]+)\s*\(([^;]*?)\)\s*(?:->[^;]*)?;", sys_rs, re.S)}
    consts = set(re.findall(r"pub const (IPCFP_[A-Z0-9_]+)", sys_rs))
    types = set(re.findall(r"pub (?:struct|type) (ipcfp_[a-z0-9_]+)", sys_rs))
    used = set(re.findall(r"sys::([A-Za-z0-9_]+)", shim))
    assert used, "the shim names no binding at all?"
    unknown = {u for u in used if u not in fns and u not in consts and u not in types}
    assert not unknown, unknown

    def n_args(text):
        depth, n, any_tok = 0, 0, False
        for ch in text:
            if ch in "([{<":
                depth += 1
            elif ch in ")]}>":
                depth -= 1
            elif ch == "," and depth == 0:
                n += 1
                continue
            if not ch.isspace():
                any_tok = True
        return (n + 1) if any_tok and not text.rstrip().endswith(",") else n

    for m in re.finditer(r"sys::(ipcfp_[a-z0-9_]+)\s*\(", shim):
        name = m.group(1)
        i, depth = m.end(), 1
        while depth:
            depth += {"(": 1, ")": -1}.get(shim[i], 0)
            i += 1
        call_args = shim[m.end():i - 1].replace("->", "")
        assert n_args(call_args) == n_args(fns[name].replace("->", "")), (name, call_args)


def test_hidden_internals_build_exports_only_the_c_abi_and_survives_a_clashing_cxx_host():
    """`make HIDE_INTERNALS=1` (linker version script csrc/exports.map): the dynamic symbol table holds exactly the functions
    include/ipcfp.h declares, and a C++ host that defines its own `ipcfp::Error` — the clash that corrupted the heap against the default
    build (DESIGN.md §7.12) — gets a clean IPCFP_ERR_NO_DEVICE / a working store. Links the objects `make` already built; CPU only."""
    import shutil
    objs = [os.path.join(ROOT, "ipc_filecoin_proofs_b200", "csrc", n) for n in os.listdir(os.path.join(ROOT, "ipc_filecoin_proofs_b200", "csrc")) if n.endswith(".o")]
    if not objs or not shutil.which("nvcc") or not shutil.which("g++"):
        import pytest
        pytest.skip("objects of libipcfp.so / nvcc / g++ not available")
    with tempfile.TemporaryDirectory() as td:
        lib = os.path.join(td, "libipcfp.so")
        subprocess.check_call(["make", "-C", ROOT, "-s", "HIDE_INTERNALS=1", f"LIB_OUT={lib}", lib])
        syms = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True, check=True).stdout.split("\n")
        exported = {l.split()[-1] for l in syms if l.strip()}
        hdr = open(os.path.join(ROOT, "include", "ipcfp.h")).read()
        declared = set(re.findall(r"\b(ipcfp_[a-z0-9_]+)\s*\(", hdr)) - {"ipcfp_store", "ipcfp_tipset"}
        assert exported == declared, (sorted(exported - declared), sorted(declared - exported))
        src = os.path.join(td, "clash.cpp")
        with open(src, "w") as f:
            f.write(r'''
#include <cstdio>
#include <string>
#include "ipcfp.h"
static int g_host_dtor_calls = 0;
namespace ipcfp {   // a host that (wrongly) defines a type where the library keeps its internal error type (csrc/common.cuh). Same layout here,
// so that being interposed is harmless and can be COUNTED: every time the library destroys one of ITS exceptions through this
// destructor, the host's symbol has replaced the library's own.
struct Error {
    int status; std::string msg; unsigned long index;
    Error(int s, std::string m, unsigned long i = ~0ul) : status(s), msg(std::move(m)), index(i) {}
    ~Error() { g_host_dtor_calls++; }
};
}
int main() {
    int no_device = 0;
    for (int k = 0; k < 50; k++) {
        ipcfp_store* s = nullptr;
        unsigned char cid[38] = {1, 0x71, 0xa0, 0xe4, 2, 0x20}, blob[8] = {0x80};
        unsigned long long off = 0;
        unsigned int len = 1;
        ipcfp_status st = ipcfp_store_create(cid, (const uint64_t*)&off, &len, blob, 1, 1, 0, 0, &s);   // without a device: throws and catches its own ipcfp::Error inside
        if (st != IPCFP_OK && st != IPCFP_ERR_NO_DEVICE) { printf("status %d\n", (int)st); return 1; }
        if (st == IPCFP_OK) ipcfp_store_destroy(s); else no_device++;
    }
    const int from_library = g_host_dtor_calls;
    try { throw ipcfp::Error(3, std::string(100, 'x')); } catch (const ipcfp::Error& e) { if (e.status != 3) return 2; }
    printf("library-internal exceptions destroyed by the HOST's destructor: %d of %d\n", from_library, no_device);
    return 0;
}
''')
        exe = os.path.join(td, "clash")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-o", exe, src, "-L" + td, "-lipcfp", "-Wl,-rpath," + td])
        out = subprocess.run([exe], capture_output=True, text=True, env=dict(os.environ, MALLOC_CHECK_="3"))
        assert out.returncode == 0 and "destroyed by the HOST's destructor: 0 of" in out.stdout, (out.returncode, out.stdout, out.stderr[-2000:])
        # the same program against the DEFAULT build shows the hazard the version script removes (only visible without a device, when the
        # library throws internally): every one of its exceptions goes through the host's destructor
        default_dir = os.path.join(ROOT, "ipc_filecoin_proofs_b200")
        exe2 = os.path.join(td, "clash_default")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-o", exe2, src, "-L" + default_dir, "-lipcfp", "-Wl,-rpath," + default_dir])
        out2 = subprocess.run([exe2], capture_output=True, text=True)
        assert out2.returncode == 0, (out2.stdout, out2.stderr[-2000:])
        n_host, n_throw = [int(x) for x in re.findall(r"(\d+) of (\d+)", out2.stdout)[0]]
        assert n_host == n_throw, out2.stdout   # documents the default build's behaviour; becomes 0 once HIDE_INTERNALS is the default
