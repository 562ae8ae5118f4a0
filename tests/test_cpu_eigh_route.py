"""`not gpu`: linalg._EIGH_LIB_MIN_BATCH (which workloads one ard_sym_eigh call solves instead of torch.linalg.eigh per matrix) is
exactly what profiles/eigh_bench.json measured: the library route is taken on a measured workload iff it was faster there."""
import json
import os

from audio_residual_b200.linalg import eigh_library_wins

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_eigh_route_table_matches_the_measurement():
    with open(os.path.join(ROOT, "profiles", "eigh_bench.json")) as f:
        res = json.load(f)
    assert "B200" in res["card"]["name"] and res["card"]["power_limit"]
    cases = [(r["batch"], r["D"], r["ard_sym_eigh_s"] < r["eigh_loop_s"]) for r in res["runs"].values()]
    cases += [(1, r["D"], r["ard_sym_eigh_s"] < r["torch_eigh_device_s"]) for r in res["single"]]
    assert len(cases) == 12
    for batch, D, wins in cases:
        assert eigh_library_wins(batch, D) == wins, (batch, D)
