"""Host logic of finalize_head_spectra's solver choice: a group of same-size heads goes to ard_sym_eigvals only from the batch where
the committed crossover sweep (profiles/eig_bench.json, tools/eig_bench.py) measured the library faster than the per-head
torch.linalg.eigvalsh loop."""
import json
import os

from audio_residual_b200.analyze_attention import _LIB_MIN_BATCH, _library_wins

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_route_follows_the_measured_crossover():
    with open(os.path.join(ROOT, "profiles", "eig_bench.json")) as f:
        sweep = json.load(f)["crossover"]
    assert {r["D"] for r in sweep} == {d for d, _ in _LIB_MIN_BATCH}
    for r in sweep:
        # routed to the library exactly where it measured faster, at every measured point past the first win too
        assert _library_wins(r["batch"], r["D"]) == r["library_wins"], r
    for d, b in _LIB_MIN_BATCH:      # both sides of every crossover are in the sweep
        assert any(r["D"] == d and r["batch"] < b and not r["library_wins"] for r in sweep)
        assert any(r["D"] == d and r["batch"] >= b and r["library_wins"] for r in sweep)


def test_sizes_between_measured_ones_take_the_larger_entry():
    assert not _library_wins(1, 4096) and not _library_wins(4, 4096) and _library_wins(8, 4096)
    assert _library_wins(4, 1000) and not _library_wins(4, 1500) and _library_wins(8, 1500)
    assert not _library_wins(4, 16) and _library_wins(8, 16)
    assert not _library_wins(4, 8192) and _library_wins(8, 8192)
