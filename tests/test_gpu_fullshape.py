"""GPU parity at the BENCHMARKED sizes (BASELINE.json configs 2-5), product vs the unmodified
reference (its stored answers, tests/golden_reference.py): per-read best score, graph-CIGAR length and FNV-1a hash of every CIGAR word,
DP-cell totals, consensus and coverage.

Small cases cannot reach what these do: 25 k-row graphs, bands wider than one 256-cell pass, scores
close to the packed kernel's int16 window, graphs past the point where the reference itself switches
to int32 (gn > 16 364), 20-pass rows in local mode.
"""
import pytest

from abpoa_b200 import synth
from abpoa_b200.batch import BatchEngine
from golden_reference import assert_batch_matches_reference

pytestmark = pytest.mark.gpu


def compare(got, ref, tag):
    assert len(got) == len(ref)
    for gi, (r, w) in enumerate(zip(got, ref)):
        assert_batch_matches_reference(r, w, f"{tag} group {gi}", msa=False)


@pytest.mark.parametrize("engine", ["chain", "launch"])
@pytest.mark.parametrize("name,n_groups", [("convex_10k", 4), ("affine_1k", 6), ("local_linear_5k", 1), ("aa_blosum62_2k", 2)])
def test_full_shape(reference_lib, name, n_groups, engine):
    """engine: the device-resident chain (default for global/banded/consensus runs) or the launch-per-round engine."""
    w = synth.WORKLOADS[name]
    if engine == "chain" and w.cfg.align_mode != 0:
        pytest.skip("local mode always takes the launch engine")
    groups = w.groups(n_groups, base_seed=4200)
    ref = reference_lib.groups(w.cfg, groups)
    with BatchEngine() as eng:
        got = eng.run(w.cfg, groups, record_reads=True, no_chain=(engine == "launch"))
        st = eng.stats()
    if engine == "chain":
        assert st["chain_groups"] == n_groups and st["chain_fallback_groups"] == 0, st
    compare(got, ref, f"{name}/{engine}")


def test_full_shape_convex_generic_kernels(reference_lib, monkeypatch):
    """The same 10 kbp x 50 shape with the packed kernel switched off: generic int16 planes while the reference's
    criterion allows (gn <= 16 364), int32 planes beyond -- both instantiations at full size."""
    monkeypatch.setenv("ABPOA_GPU_NO_P16", "1")
    w = synth.WORKLOADS["convex_10k"]
    groups = w.groups(1, base_seed=4300)
    ref = reference_lib.groups(w.cfg, groups)
    with BatchEngine(n_workers=1, groups_per_launch=1) as eng:
        got = eng.run(w.cfg, groups, record_reads=True)
    compare(got, ref, "convex_10k/generic")
