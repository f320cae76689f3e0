"""tests/host_fuzz/emu_multi.cu: the per-item device code of ipcfp_generate_event_proof_multi — `pass1_multi_decode`
(`event_spec_mask`, `node_events_multi`, `walk_events_multi`), `pair_count_item`, `pass2_multi_item` (csrc/events_items.cuh,
csrc/ipld.cuh) — compiled for the host and driven item by item over a host copy of the store, against the oracle's
generate_proof_bundle with the same event specs: per-spec matching receipts, every EventProof field, the union witness, n_exec; and,
with one block mutated under its CID or missing (half of them blocks that only a later spec's matches reach), the same status at
the same index. Honours IPCFP_HOST_FUZZ_SANITIZE=1 (AddressSanitizer + UBSan, no reports allowed)."""
import subprocess

from tests.test_host_fuzz import _harness


def test_multi_spec_path_emulated_on_cpu_matches_oracle_bundle():
    exe, env = _harness("emu_multi", with_synth=True)
    out = subprocess.run([exe, "24", "60", "7"], capture_output=True, text=True, env=env)
    assert out.returncode == 0, (out.stdout + out.stderr)[-3000:]
    assert out.stdout.startswith("ok: multi-spec event path on the CPU == oracle bundle for 24 tipsets"), out.stdout
    assert "runtime error" not in out.stderr and "AddressSanitizer" not in out.stderr, out.stderr[-3000:]
    runs_ok, runs_err = int(out.stdout.split(":")[2].split()[0]), int(out.stdout.split("field,")[1].split()[0])
    later = int(out.stdout.split("identically,")[1].split()[0])
    assert runs_ok > 100 and runs_err > 500 and later > 200, out.stdout
