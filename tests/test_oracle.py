"""CPU suite, part 1: pin the oracle.

* the scalar restatement (oracle/poa_oracle.c) reproduces the golden vectors generated from
  the unmodified reference (tests/golden/golden.json, made by tests/golden/make_golden.py);
* it is also compared, read by read, with the reference's stored answers for more groups
  (tests/golden_reference.py: scores, CIGAR words, end points, DP-cell counts).
The alignments come from the oracle; graph fusion / consensus / MSA run in the product's host
layer, so this also pins that layer on the CPU.
"""
import json
from pathlib import Path

import pytest

from abpoa_b200.aligner import PoaConfig
from cases import CASES, case_reads, case_weights
from helpers import assert_digest_equal, assert_group_equal, group_digest, run_group

GOLDEN = json.loads((Path(__file__).parent / "golden" / "golden.json").read_text())


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_matches_golden(product_lib, name):
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    reads = case_reads(case)
    got = group_digest(run_group(product_lib, cfg, reads, use_oracle=True, weights=case_weights(case, reads)), cfg.m)
    assert_digest_equal(got, GOLDEN["cases"][name], name)


@pytest.mark.parametrize("name", ["seq_affine", "syn_convex_2k", "syn_local_linear", "syn_aa_blosum62", "syn_ragged"])
def test_oracle_matches_live_reference(product_lib, reference_lib, name):
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    reads = case_reads(case)
    assert_group_equal(run_group(product_lib, cfg, reads, use_oracle=True), run_group(reference_lib, cfg, reads), name)


GLOBAL_CASES = [n for n, c in CASES.items() if c["cfg"].get("align_mode", 0) == 0]


@pytest.mark.parametrize("name", GLOBAL_CASES)
def test_spliced_order_matches_golden(product_lib, name):
    """Global mode: the batch engine keeps the previous topological order and splices the new nodes
    in instead of re-running the Kahn pass per read (poa_graph.c "spliced order").  Every alignment
    (score, graph-CIGAR in node ids, end points, DP cells), consensus and RC-MSA must be unchanged."""
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    reads = case_reads(case)
    r = run_group(product_lib, cfg, reads, use_oracle=True, fast_order=True, weights=case_weights(case, reads))
    spliced, fallback = r["order_stats"]
    assert spliced > 0 and fallback == 0, (spliced, fallback)
    assert_digest_equal(group_digest(r, cfg.m), GOLDEN["cases"][name], name)


@pytest.mark.parametrize("name", GLOBAL_CASES)
def test_consensus_only_mode_matches_golden(product_lib, name):
    """Consensus-only runs (no RC-MSA, hence no per-edge read sets) take the host's fast paths: the
    heaviest-edge shortcut of the fusion loop and the spliced topological order.  Alignments, consensus
    and coverage must equal the golden vectors (which were generated with the MSA on)."""
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    reads = case_reads(case)
    r = run_group(product_lib, cfg, reads, want_msa=False, use_oracle=True, fast_order=True, weights=case_weights(case, reads))
    got, want = group_digest(r, cfg.m), GOLDEN["cases"][name]
    assert len(got["alns"]) == len(want["alns"])
    for i, (x, y) in enumerate(zip(got["alns"], want["alns"])):
        assert x == y, f"{name} read {i}: {x} != {y}"
    assert got["cons"] == want["cons"] and got["cov_sha1"] == want["cov_sha1"], name


def test_linear_banded_decisions_match_reference(product_lib, reference_lib):
    """Global banded linear-gap alignment: the reference's AVX2 row procedure leaks H[end]-k*E1 into the
    last vector of a row (SURVEY 8a a7), the restatement follows the textbook recurrence.  The leaked
    cells never changed a decision: scores and graph-CIGARs are identical on a sweep of group shapes,
    error rates (3-25 %) and band widths."""
    from cases import LINEAR
    from abpoa_b200 import synth
    n_aln = 0
    for seed in range(60):
        reads = synth.make_group(5000 + seed, 4 + seed % 5, 150 + 37 * (seed % 9), [0.03, 0.08, 0.15, 0.25][seed % 4])
        cfg = PoaConfig(**LINEAR) if seed % 2 == 0 else PoaConfig(wb=6 + seed % 7, wf=0.01, **LINEAR)
        a = run_group(product_lib, cfg, reads, use_oracle=True)
        # every score, graph-CIGAR, end point and the band of every row (hence the cell count): exact since the
        # restatement follows the vector procedure lane for lane; consensus, coverage and RC-MSA as well
        assert_group_equal(a, run_group(reference_lib, cfg, reads), f"linear banded seed {seed}")
        n_aln += sum(1 for x in a["alns"] if x.aligned)
    assert n_aln >= 250
    print(f"banded linear: {n_aln} alignments")


@pytest.mark.parametrize("shape", [(301, 14, 4000, 0.10), (302, 25, 1500, 0.20), (303, 40, 600, 0.30)])
def test_spliced_order_on_bushy_graphs_vs_live_reference(product_lib, reference_lib, shape):
    """Deeper groups with high error rates grow large aligned-node groups and long insertion chains --
    the cases the splice rules (anchor behind the whole aligned group, inherited anchors) exist for.
    Every alignment, the consensus and the RC-MSA must equal the live reference, with no fallback to
    the full Kahn pass."""
    from abpoa_b200 import synth
    seed, n, length, err = shape
    reads = synth.make_group(seed, n, length, err)
    cfg = PoaConfig()
    a = run_group(product_lib, cfg, reads, use_oracle=True, fast_order=True)
    spliced, fallback = a["order_stats"]
    assert spliced >= n - 2 and fallback == 0, (spliced, fallback)
    assert_group_equal(a, run_group(reference_lib, cfg, reads), f"bushy {shape}")
