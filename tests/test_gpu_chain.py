"""GPU parity of the device-resident chain engine (poa_chain.cu / poa_chain.cuh): the whole progressive
loop of a group -- align, fuse, re-order, flatten -- runs on the GPU; results must equal the unmodified
reference group by group (per-read score, CIGAR length and FNV-1a hash, DP cells, consensus, coverage),
and groups the device cannot finish must come back through the launch engine with the same results."""
import numpy as np
import pytest

from abpoa_b200 import synth
from abpoa_b200.aligner import PoaConfig
from abpoa_b200.batch import BatchEngine
from cases import AFFINE
from golden_reference import assert_batch_matches_reference
from helpers import run_group

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["free-running", "rounds"])
def chain_mode(request, monkeypatch):
    """Every test runs on both schedules of the chain engine: free-running groups (two persistent kernels, the default) and
    lock-step rounds (two kernels per round and cohort)."""
    if request.param == "rounds":
        monkeypatch.setenv("ABPOA_GPU_CHAIN_ROUNDS", "1")
    else:
        monkeypatch.delenv("ABPOA_GPU_CHAIN_ROUNDS", raising=False)
    return request.param


def check(reference_lib, cfg, groups, expect_chain=None, expect_fallback=None, **engine_kw):
    with BatchEngine(**engine_kw) as eng:
        got = eng.run(cfg, groups, record_reads=True)
        st = eng.stats()
    for gi, (g, r) in enumerate(zip(groups, got)):
        ref = run_group(reference_lib, cfg, g, want_msa=False)
        assert r.n_aligned == max(len(g) - 1, 0) or len(g) == 0, f"group {gi}: n_aligned"
        assert_batch_matches_reference(r, ref, f"group {gi}", msa=False)
    if expect_chain is not None:
        assert st["chain_groups"] == expect_chain, st
    if expect_fallback is not None:
        assert st["chain_fallback_groups"] == expect_fallback, st
    return st


@pytest.mark.parametrize("gap", ["convex", "affine"])
def test_chain_many_groups(reference_lib, gap):
    kw = {} if gap == "convex" else AFFINE
    groups = [synth.make_group(5000 + g, 6 + g % 5, 300 + 40 * (g % 7), 0.04 + 0.01 * (g % 6)) for g in range(40)]
    check(reference_lib, PoaConfig(**kw), groups, expect_chain=40, expect_fallback=0)


def test_chain_ragged_and_degenerate_groups(reference_lib):
    """Groups of very different sizes in one call, reads of very different lengths inside a group, a single-read
    group and an empty group (both never reach the chain), a 2-read group."""
    rng = np.random.default_rng(5)
    groups = []
    for g in range(12):
        base = synth.make_group(5200 + g, 3 + 2 * (g % 5), 900, 0.06)
        groups.append([np.ascontiguousarray(r[: int(rng.integers(5, len(r)))]) if (i % 3 == 1) else r for i, r in enumerate(base)])
    groups.append(synth.make_group(5300, 2, 500, 0.05))
    groups.append(synth.make_group(5301, 1, 100, 0.0))
    groups.append([])
    st = check(reference_lib, PoaConfig(), groups)
    assert st["chain_groups"] >= 12


def test_chain_high_error_deep(reference_lib):
    """25 % error, 30 reads: many new nodes per read, aligned sets of full size, long insertion chains."""
    groups = [synth.make_group(5400 + g, 30, 500, 0.25) for g in range(4)]
    check(reference_lib, PoaConfig(), groups)


def test_chain_amino_acid(reference_lib):
    cfg = synth.WORKLOADS["aa_blosum62_2k"].cfg
    groups = [synth.make_group(5500 + g, 12, 600, 0.10, m=27) for g in range(8)]
    check(reference_lib, cfg, groups, expect_chain=8, expect_fallback=0)


def test_chain_hands_back_groups_it_cannot_finish(reference_lib, monkeypatch):
    """Two edge slots per node: most groups outgrow their device slot, are reported back and finished by the
    launch engine -- with identical results."""
    monkeypatch.setenv("ABPOA_GPU_CHAIN_K", "2")
    groups = [synth.make_group(5600 + g, 8, 400, 0.10) for g in range(10)]
    st = check(reference_lib, PoaConfig(), groups)
    assert st["chain_fallback_groups"] > 0 and st["chain_groups"] + st["chain_fallback_groups"] == 10


def test_chain_single_cohort_and_many_cohorts(reference_lib, monkeypatch):
    groups = [synth.make_group(5700 + g, 7, 350, 0.05) for g in range(9)]
    for c in ("1", "16"):
        monkeypatch.setenv("ABPOA_GPU_CHAIN_COHORTS", c)
        check(reference_lib, PoaConfig(**AFFINE), groups, expect_chain=9, expect_fallback=0)


def test_chain_and_launch_engine_agree(reference_lib):
    """Same call with and without the chain: identical records."""
    groups = [synth.make_group(5800 + g, 10, 700, 0.07) for g in range(6)]
    cfg = PoaConfig()
    with BatchEngine() as eng:
        a = eng.run(cfg, groups, record_reads=True)
        sa = eng.stats()
        eng.reset_stats()
        b = eng.run(cfg, groups, record_reads=True, no_chain=True)
        sb = eng.stats()
    assert sa["chain_groups"] == 6 and sb["chain_groups"] == 0
    for x, y in zip(a, b):
        assert x.dp_cells == y.dp_cells
        assert np.array_equal(x.read_best_score[1:], y.read_best_score[1:]) and np.array_equal(x.read_cigar_hash[1:], y.read_cigar_hash[1:])
        assert all(np.array_equal(p, q) for p, q in zip(x.cons, y.cons)) and all(np.array_equal(p, q) for p, q in zip(x.cov, y.cov))


def test_chain_graph_export_cross_check(reference_lib, monkeypatch):
    """ABPOA_GPU_CHAIN_EXPORT_GRAPH=1: instead of the device's consensus the whole device-built graph comes back and the
    host layer computes the consensus on it -- both routes must agree with the reference."""
    groups = [synth.make_group(5900 + g, 9, 450, 0.08) for g in range(6)]
    check(reference_lib, PoaConfig(), groups, expect_chain=6, expect_fallback=0)
    monkeypatch.setenv("ABPOA_GPU_CHAIN_EXPORT_GRAPH", "1")
    check(reference_lib, PoaConfig(), groups, expect_chain=6, expect_fallback=0)


def test_chain_more_groups_than_resident_warps(reference_lib, chain_mode):
    """1600 tiny groups: more than the alignment warps one B200 keeps resident (9 per SM), so late groups start when early ones
    have left; the fuse queue sees every group several times."""
    groups = [synth.make_group(6000 + g, 3 + g % 3, 60 + g % 50, 0.06) for g in range(1600)]
    st = check(reference_lib, PoaConfig(**AFFINE), groups, expect_chain=1600, expect_fallback=0)
    assert st["chain_free_running"] == (1 if chain_mode == "free-running" else 0)
