"""GPU parity, part 2: every named case of tests/cases.py through the CUDA kernels.

* single-alignment path (abpoa.h: abpoa_align_sequence_to_graph + abpoa_add_graph_alignment) against
  the golden vectors generated from the unmodified reference (tests/golden/golden.json) -- no oracle,
  no reference library involved: per-read score, CIGAR sha1, end points, DP cells, consensus, RC-MSA;
* batch engine (abpoa_gpu.h) against the reference's stored answers (tests/golden_reference.py) with per-read CIGAR hashes;
* every fallback of the launcher forced through environment switches: generic int16 kernel
  (ABPOA_GPU_NO_P16), range guard of the packed kernel (ABPOA_GPU_FORCE_P16 on a case that needs 32
  bits), plane-slab overflow redo (ABPOA_GPU_SLAB_PCT), Kahn order instead of the spliced order
  (ABPOA_GPU_EXACT_ORDER), plane-arena contention in the pipelined engine (ABPOA_GPU_ARENA_MB);
* graph shapes the synthetic sets never produce: > 32 predecessors of one node;
* the remaining entry points of the path: strand retry (-s) and sub-graph alignment (+ -G).
"""
import ctypes as C
import json
from pathlib import Path

import numpy as np
import pytest

from abpoa_b200 import capi, synth
from abpoa_b200.aligner import PoaConfig, PoaSession
from abpoa_b200.batch import BatchEngine
from abpoa_b200.capi import abpoa_res_t, c_u8_p
from cases import AFFINE, CASES, case_reads, case_weights
from golden_reference import GoldenReference, arrays_digest, assert_batch_matches_reference, digest
from helpers import assert_digest_equal, assert_group_equal, group_digest, run_group

pytestmark = pytest.mark.gpu

GOLDEN = json.loads((Path(__file__).parent / "golden" / "golden.json").read_text())


def digest_vs_golden(lib, name, strip_cells=False):
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    reads = case_reads(case)
    got = group_digest(run_group(lib, cfg, reads, weights=case_weights(case, reads)), cfg.m)
    want = json.loads(json.dumps(GOLDEN["cases"][name]))
    if strip_cells:
        for a in got["alns"] + want["alns"]:
            a.pop("cells", None)
    assert_digest_equal(got, want, name)


@pytest.mark.parametrize("name", list(CASES))
def test_case_vs_golden(product_lib, name):
    digest_vs_golden(product_lib, name)


NO_P16_CASES = ["seq_affine", "heter_convex", "syn_affine_1k", "syn_convex_2k", "syn_linear_banded", "syn_local_linear", "syn_local_affine",
                "syn_extend_convex_zdrop", "syn_aa_blosum62", "syn_path_score", "syn_gap_on_right", "syn_ragged"]


@pytest.mark.parametrize("name", NO_P16_CASES)
def test_generic_int16_kernel(product_lib, monkeypatch, name):
    """ABPOA_GPU_NO_P16=1: the 32-bit-register kernel with int16 planes (the fallback of the packed kernel)."""
    monkeypatch.setenv("ABPOA_GPU_NO_P16", "1")
    digest_vs_golden(product_lib, name)


def _retries(session):
    fn = session.lib.dll.poa_debug_retries
    fn.restype = C.c_int64
    fn.argtypes = [capi.abpoa_t_p]
    return fn(session.ab)


def run_group_counting_retries(lib, cfg, reads):
    cfg = PoaConfig(**{**cfg.__dict__, "out_msa": True})
    with PoaSession(cfg, lib) as s:
        alns = s.run_reads(reads)
        s.generate()
        return {"alns": alns, "cons": s.consensus(), "cov": s.consensus_cov(), "msa": s.msa_rows(), "order_stats": None}, _retries(s)


def test_range_guard_redo(product_lib, reference_lib, monkeypatch):
    """Scores that really leave the int16 window (2 kbp x match 20 = 40 000), forced onto the packed int16 kernel: its
    run-time guard must report POA_ST_RANGE and the 32-bit redo must give the reference's result."""
    monkeypatch.setenv("ABPOA_GPU_FORCE_P16", "1")
    cfg = PoaConfig(**CASES["syn_convex_int32"]["cfg"])
    reads = synth.make_group(31, 6, 2000, 0.05)
    got, retries = run_group_counting_retries(product_lib, cfg, reads)
    assert retries > 0, "the packed kernel never reported RANGE on scores beyond int16"
    assert_group_equal(got, run_group(reference_lib, cfg, reads), "range-redo")


@pytest.mark.parametrize("name", ["syn_convex_2k", "syn_affine_1k", "syn_high_error"])
def test_plane_overflow_redo(product_lib, monkeypatch, name):
    """A plane slab far smaller than the band needs: POA_ST_PLANE_OVF, then the full-rectangle redo."""
    monkeypatch.setenv("ABPOA_GPU_SLAB_PCT", "30")
    case = CASES[name]
    cfg = PoaConfig(**case["cfg"])
    got, retries = run_group_counting_retries(product_lib, cfg, case_reads(case))
    assert retries > 0, "the slab never overflowed: the hook did not bite"
    assert_digest_equal(group_digest(got, cfg.m), GOLDEN["cases"][name], "plane-ovf-redo")


# ------------------------------------------------------------------------------------------- batch engine
def check_batch(reference_lib, cfg, groups, weights=None, cells=True, **engine_kw):
    with BatchEngine(**engine_kw) as eng:
        got = eng.run(cfg, groups, record_reads=True, weights=weights)
        st = eng.stats()
    assert st["alignments"] >= sum(max(len(g) - 1, 0) for g in groups)
    for gi, (g, r) in enumerate(zip(groups, got)):
        ref = run_group(reference_lib, cfg, g, want_msa=cfg.out_msa, weights=weights[gi] if weights else None)
        assert_batch_matches_reference(r, ref, f"group {gi}", cells=cells)
    return st


@pytest.mark.parametrize("name", list(CASES))
def test_case_batch_engine(reference_lib, name):
    """The same cases through abpoa_gpu_msa_batch (two groups: the case's reads, and the same reads in
    reverse order so that the groups differ), alternately consensus-only and with the RC-MSA."""
    case = CASES[name]
    want_msa = (list(CASES).index(name) % 2) == 0
    cfg = PoaConfig(**{**case["cfg"], "out_msa": want_msa})
    reads = case_reads(case)
    w = case_weights(case, reads)
    groups = [reads, reads[::-1]]
    weights = [w, w[::-1]] if w is not None else None
    check_batch(reference_lib, cfg, groups, weights=weights, n_workers=2, groups_per_launch=1)


def test_batch_exact_order(reference_lib, monkeypatch):
    """ABPOA_GPU_EXACT_ORDER=1: the reference's Kahn order after every read instead of the spliced order."""
    monkeypatch.setenv("ABPOA_GPU_EXACT_ORDER", "1")
    groups = [synth.make_group(1300 + g, 6, 500, 0.08) for g in range(6)]
    check_batch(reference_lib, PoaConfig(), groups, n_workers=2, groups_per_launch=2)


def test_batch_arena_contention(reference_lib, monkeypatch):
    """A plane arena that holds only a few launches: sub-chunks must take the drain-then-block path
    (no worker waits for planes while holding some) and still deliver every group."""
    monkeypatch.setenv("ABPOA_GPU_ARENA_MB", "4")
    groups = [synth.make_group(1500 + g, 8, 300 + 20 * (g % 5), 0.05) for g in range(64)]
    check_batch(reference_lib, PoaConfig(**AFFINE), groups, n_workers=4, groups_per_launch=4)


def test_batch_no_p16_and_slab_redo(reference_lib, monkeypatch):
    """Redo paths inside the pipelined engine (poa_engine_collect): slab overflow on the generic kernel (with the packed
    kernel switched off the chain engine, which only has that kernel, steps aside)."""
    monkeypatch.setenv("ABPOA_GPU_NO_P16", "1")
    monkeypatch.setenv("ABPOA_GPU_SLAB_PCT", "30")
    groups = [synth.make_group(1700 + g, 6, 400, 0.06) for g in range(10)]
    st = check_batch(reference_lib, PoaConfig(), groups, n_workers=2, groups_per_launch=3)
    assert st["retries"] > 0


# ------------------------------------------------------------------------------------------- graph shapes
def deletion_fan(seed=7, n=40, flank=220):
    """Reads that delete 1..n-1 bases in front of the same template position: that node collects one
    in-edge per read (> 32 predecessors: the chunked predecessor loops of the DP and of the backtrace)."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 4, size=2 * flank).astype(np.uint8)
    return [t] + [np.concatenate([t[: flank - k], t[flank:]]) for k in range(1, n)]


@pytest.mark.parametrize("gap", ["convex", "affine"])
def test_more_than_32_predecessors(product_lib, reference_lib, gap):
    cfg = PoaConfig(**(AFFINE if gap == "affine" else {}))
    reads = deletion_fan()
    ref = run_group(reference_lib, cfg, reads)

    def max_in_degree(lib):
        with PoaSession(cfg, lib) as s:
            s.run_reads(reads, count_cells=False)
            g = s.ab.contents.abg.contents
            return max(g.node[i].in_edge_n for i in range(g.node_n))
    deg = reference_lib.value("max_in_degree", (cfg.__dict__, reads), max_in_degree)
    assert deg > 32, f"the construction only reached in-degree {deg}"
    assert_group_equal(run_group(product_lib, cfg, reads), ref, f"fan/{gap}")


def test_more_than_32_predecessors_generic_kernel(product_lib, reference_lib, monkeypatch):
    monkeypatch.setenv("ABPOA_GPU_NO_P16", "1")
    cfg = PoaConfig()
    reads = deletion_fan(seed=8)
    assert_group_equal(run_group(product_lib, cfg, reads), run_group(reference_lib, cfg, reads), "fan/generic")


# ------------------------------------------------------------------------------------------- -s and sub-graphs
def strand_mix(seed, n, length):
    reads = synth.make_group(seed, n, length, 0.05)
    out = []
    for i, r in enumerate(reads):
        out.append(np.ascontiguousarray((3 - r)[::-1]) if i % 3 == 1 else r)   # every third read arrives reverse-complemented
    return out


def msa_whole(lib, cfg, reads):
    """abpoa_msa over the whole group: which reads were flipped, digests of consensus, coverage and RC-MSA
    (for the stored reference: its stored answer)."""
    def run(lib):
        with PoaSession(cfg, lib) as s:
            s.msa(reads)
            abs_ = s.ab.contents.abs.contents
            is_rc = [int(abs_.is_rc[i]) for i in range(len(reads))]
            return {"cons": arrays_digest(s.consensus()), "cov": arrays_digest(s.consensus_cov()), "msa": arrays_digest(s.msa_rows()), "is_rc": is_rc}
    if isinstance(lib, GoldenReference):
        return lib.value("msa_whole", (cfg.__dict__, reads), run)
    return run(lib)


def test_amb_strand_msa(product_lib, reference_lib):
    """abpoa_msa with -s (reference src/abpoa_align.c:323-344): weak forward hits are re-aligned as reverse complement."""
    cfg = PoaConfig(amb_strand=True, out_msa=True)
    reads = strand_mix(1900, 9, 600)
    a, b = msa_whole(product_lib, cfg, reads), msa_whole(reference_lib, cfg, reads)
    assert sum(b["is_rc"]) >= 2, "the reference flipped no read: the case does not exercise -s"
    assert a["is_rc"] == b["is_rc"]
    assert a["cons"] == b["cons"]
    assert a["msa"] == b["msa"]


def test_amb_strand_batch(product_lib, reference_lib):
    cfg = PoaConfig(amb_strand=True, out_msa=True)
    groups = [strand_mix(1950 + g, 7, 400 + 50 * g) for g in range(5)]
    with BatchEngine(n_workers=2, groups_per_launch=2) as eng:
        got = eng.run(cfg, groups)
    for gi, (g, r) in enumerate(zip(groups, got)):
        ref = msa_whole(reference_lib, cfg, g)
        assert arrays_digest(r.cons) == ref["cons"], f"group {gi}: consensus"
        assert arrays_digest(r.msa) == ref["msa"], f"group {gi}: msa"


def subgraph_walk(lib, cfg, reads, windows):
    """The loop of the reference's sub_example.c: read i is aligned to the sub-graph between the nodes
    that enclose [inc_beg, inc_end] (abpoa_subgraph_nodes) and fused with abpoa_add_subgraph_alignment.
    Per read (rc, window begin, window end, score, digest of the graph-CIGAR, end points), digests of the
    consensus and the RC-MSA (for the stored reference: its stored answer)."""
    if isinstance(lib, GoldenReference):
        return lib.value("subgraph_walk", (cfg.__dict__, reads, windows), lambda live: subgraph_walk(live, cfg, reads, windows))
    d = lib.dll
    d.abpoa_subgraph_nodes.argtypes = [capi.abpoa_t_p, capi.abpoa_para_t_p, C.c_int, C.c_int, capi.c_int_p, capi.c_int_p]
    d.abpoa_align_sequence_to_subgraph.restype = C.c_int
    d.abpoa_align_sequence_to_subgraph.argtypes = [capi.abpoa_t_p, capi.abpoa_para_t_p, C.c_int, C.c_int, c_u8_p, C.c_int, C.POINTER(abpoa_res_t)]
    d.abpoa_add_subgraph_alignment.argtypes = [capi.abpoa_t_p, capi.abpoa_para_t_p, C.c_int, C.c_int, c_u8_p, capi.c_int_p, C.c_int, capi.c_int_p,
                                               abpoa_res_t, C.c_int, C.c_int, C.c_int]
    out = []
    with PoaSession(cfg, lib) as s:
        s.reset(max(len(r) for r in reads))
        s.ab.contents.abs.contents.n_seq = len(reads)
        for i, (r, (wb, we)) in enumerate(zip(reads, windows)):
            r = np.ascontiguousarray(r, dtype=np.uint8)
            res = abpoa_res_t()
            eb, ee = C.c_int(0), C.c_int(1)
            if i:
                d.abpoa_subgraph_nodes(s.ab, s.abpt, wb, we, C.byref(eb), C.byref(ee))
            rc = d.abpoa_align_sequence_to_subgraph(s.ab, s.abpt, eb.value, ee.value, r.ctypes.data_as(c_u8_p), len(r), C.byref(res))
            cig = np.ctypeslib.as_array(res.graph_cigar, shape=(res.n_cigar,)).copy() if res.n_cigar > 0 else np.zeros(0, dtype=np.uint64)
            out.append([rc, eb.value, ee.value, int(res.best_score) if rc >= 0 else 0, digest(cig), [res.node_s, res.node_e, res.query_s, res.query_e] if rc >= 0 else None])
            d.abpoa_add_subgraph_alignment(s.ab, s.abpt, eb.value, ee.value, r.ctypes.data_as(c_u8_p), None, len(r), None, res, i, len(reads), 0)
            if res.n_cigar > 0:
                capi.libc_free(res.graph_cigar)
        s.generate()
        return [out, arrays_digest(s.consensus()), arrays_digest(s.msa_rows())]


@pytest.mark.parametrize("path_score", [False, True])
def test_subgraph_alignment(product_lib, reference_lib, path_score):
    """Sub-graph windows (the index_map / live-row filter of the DP entry, reference
    src/abpoa_align_simd.c:1257-1269), with and without -G, whose score lookup uses the filtered index."""
    rng = np.random.default_rng(77)
    full = synth.make_group(2100, 4, 400, 0.06)
    reads = list(full)
    windows = [(0, 1)] * len(full)
    t = full[0]
    for k in range(6):                       # partial reads aligned inside a window of node ids of the first read
        a = int(rng.integers(10, 150)); b = int(rng.integers(250, 390))
        piece = t[a:b].copy()
        piece[::17] = (piece[::17] + 1) % 4
        reads.append(piece)
        windows.append((2 + a, 2 + b - 1))   # the first read's base i became node id 2 + i
    cfg = PoaConfig(inc_path_score=path_score, out_msa=True)
    a = subgraph_walk(product_lib, cfg, reads, windows)
    b = subgraph_walk(reference_lib, cfg, reads, windows)
    assert len(a[0]) == len(b[0])
    for i, (x, y) in enumerate(zip(a[0], b[0])):
        assert x[:4] == y[:4], f"read {i}: rc / window / score {x[:4]} vs {y[:4]}"
        assert x[4] == y[4], f"read {i}: graph-CIGAR"
        assert x[5] == y[5], f"read {i}: ends"
    assert a[1] == b[1]
    assert a[2] == b[2]


# ------------------------------------------------------------------------------------------- a7: banded linear gaps, lane-exact
@pytest.mark.parametrize("mode", [0, 2])
def test_linear_banded_lane_exact_sweep(product_lib, reference_lib, mode):
    """Banded linear-gap alignment (global and extend): the specification is the reference's vector procedure (SURVEY 8a a7:
    leaked cells right of `end`, vector-granular predecessor reads, incomplete scans beyond the predecessors' last vector).
    Sweep of group shapes, error rates (3-25 %) and band widths: every score, graph-CIGAR word, end point AND the DP-cell
    count (= the band of every row) must equal the live reference."""
    from cases import LINEAR
    n_aln = 0
    for seed in range(60):
        reads = synth.make_group(5000 + seed, 4 + seed % 5, 150 + 37 * (seed % 9), [0.03, 0.08, 0.15, 0.25][seed % 4])
        cfg = PoaConfig(align_mode=mode, **LINEAR) if seed % 2 == 0 else PoaConfig(align_mode=mode, wb=6 + seed % 7, wf=0.01, **LINEAR)
        a = run_group(product_lib, cfg, reads)
        b = run_group(reference_lib, cfg, reads)
        assert_group_equal(a, b, f"linear banded mode {mode} seed {seed}")
        n_aln += sum(1 for x in a["alns"] if x.aligned)
    assert n_aln >= 250


def test_linear_banded_int32_width(product_lib, reference_lib):
    """The same with scores that make the reference pick int32 (vectors of 8 lanes instead of 16)."""
    cfg = PoaConfig(match=20, mismatch=40, gap_open1=0, gap_ext1=20, gap_open2=0, gap_ext2=0, wb=8)
    for seed in range(6):
        reads = synth.make_group(5100 + seed, 6, 1800, 0.10)
        assert_group_equal(run_group(product_lib, cfg, reads), run_group(reference_lib, cfg, reads), f"linear banded int32 seed {seed}")
