"""GPU parity of the batched engine (include/abpoa_gpu.h): many groups advanced concurrently
must give, group by group, exactly what the reference gives for abpoa_msa() on that group --
per-read best score, CIGAR length and FNV hash of the CIGAR words, DP cells, consensus,
coverage and RC-MSA."""
import pytest

from abpoa_b200 import synth
from abpoa_b200.aligner import PoaConfig
from abpoa_b200.batch import BatchEngine
from cases import AFFINE, LINEAR
from abpoa_b200.capi import ABPOA_LOCAL_MODE
from golden_reference import assert_batch_matches_reference
from helpers import run_group

pytestmark = pytest.mark.gpu


def check_batch(reference_lib, cfg, groups, **engine_kw):
    with BatchEngine(**engine_kw) as eng:
        got = eng.run(cfg, groups, record_reads=True)
        st = eng.stats()
    assert st["alignments"] == sum(max(len(g) - 1, 0) for g in groups)
    for gi, (g, r) in enumerate(zip(groups, got)):
        ref = run_group(reference_lib, cfg, g, want_msa=cfg.out_msa)
        assert_batch_matches_reference(r, ref, f"group {gi}")


def test_batch_affine_many_groups(reference_lib):
    cfg = PoaConfig(**AFFINE)
    groups = [synth.make_group(500 + g, 8, 300 + 20 * (g % 5), 0.05) for g in range(70)]
    check_batch(reference_lib, cfg, groups, n_workers=4, groups_per_launch=8)


def test_batch_convex_msa_ragged(reference_lib):
    cfg = PoaConfig(out_msa=True)
    groups = [synth.make_group(700 + g, 3 + (g % 6), 200 + 150 * (g % 4), 0.06) for g in range(23)]
    groups.append([])                                     # empty group
    groups.append(synth.make_group(9, 1, 100, 0.0))       # single read: no DP at all
    check_batch(reference_lib, cfg, groups, n_workers=3, groups_per_launch=5)


def test_batch_local_linear(reference_lib):
    cfg = PoaConfig(align_mode=ABPOA_LOCAL_MODE, **LINEAR)
    groups = [synth.make_group(900 + g, 5, 400, 0.05) for g in range(12)]
    check_batch(reference_lib, cfg, groups, n_workers=2, groups_per_launch=4)


def test_batch_amino_acid(reference_lib):
    cfg = synth.WORKLOADS["aa_blosum62_2k"].cfg
    groups = [synth.make_group(1100 + g, 6, 500, 0.10, m=27) for g in range(10)]
    check_batch(reference_lib, cfg, groups, n_workers=2, groups_per_launch=4)


@pytest.mark.parametrize("which", ["affine", "convex_msa_ragged"])
def test_batch_resident_engine(reference_lib, monkeypatch, which):
    """The opt-in resident-kernel engine (ABPOA_GPU_RESIDENT=1: one slot per group, mailboxes in
    mapped pinned memory, no launch per alignment) must give the same per-read results."""
    monkeypatch.setenv("ABPOA_GPU_RESIDENT", "1")
    monkeypatch.setenv("ABPOA_GPU_RESIDENT_BUDGET_S", "120")
    if which == "affine":
        cfg = PoaConfig(**AFFINE)
        groups = [synth.make_group(500 + g, 8, 300 + 20 * (g % 5), 0.05) for g in range(70)]
        check_batch(reference_lib, cfg, groups, n_workers=4)
    else:
        cfg = PoaConfig(out_msa=True)
        groups = [synth.make_group(700 + g, 3 + (g % 6), 200 + 150 * (g % 4), 0.06) for g in range(23)]
        groups.append([])
        groups.append(synth.make_group(9, 1, 100, 0.0))
        check_batch(reference_lib, cfg, groups, n_workers=3)
