"""Shared test helpers (pure Python, no alignment logic)."""
from __future__ import annotations

from pathlib import Path

import numpy as np

from abpoa_b200.aligner import PoaConfig, PoaSession, encode

INPUTS = Path(__file__).resolve().parent / "golden" / "inputs"


def read_fasta(path: Path, m: int = 5) -> list[np.ndarray]:
    seqs, cur = [], []
    lines = Path(path).read_text().splitlines()
    is_fq = lines and lines[0].startswith("@")
    if is_fq:
        return [encode(lines[i + 1], m) for i in range(0, len(lines) - 1, 4)]
    for ln in lines:
        if ln.startswith(">"):
            if cur:
                seqs.append(encode("".join(cur), m))
            cur = []
        elif ln.strip():
            cur.append(ln.strip())
    if cur:
        seqs.append(encode("".join(cur), m))
    return seqs


def run_group(lib, cfg: PoaConfig, reads, want_msa: bool = True, use_oracle: bool = False, fast_order: bool = False, weights=None):
    """Progressive POA of one group through `lib`; returns per-read records + consensus (+ MSA).

    use_oracle=True: the graph / consensus / MSA code of `lib` is driven, but every
    alignment comes from the scalar oracle (oracle/libpoa_oracle.so).  That is how the
    CPU-only suite exercises the product's host layer without a GPU -- a test harness
    arrangement, not a product path.

    `lib` may be the stored reference (golden_reference.GoldenReference): the result is then the
    reference's digest of the same run (compare it with assert_group_equal)."""
    from golden_reference import GoldenReference
    if isinstance(lib, GoldenReference):
        assert not use_oracle and not fast_order
        return lib.group(cfg, reads, want_msa, weights)
    cfg = PoaConfig(**{**cfg.__dict__, "out_msa": want_msa})
    with PoaSession(cfg, lib) as s:
        if use_oracle:
            from oracle_binding import oracle_align
            s.reset(max((len(r) for r in reads), default=1024))
            if fast_order:      # what the batch engine does per handle: spliced topological order between reads
                s.lib.dll.poa_graph_set_fast_order(s.ab.contents.abg, 1)
            alns = []
            for i, r in enumerate(reads):
                a, res = oracle_align(s, r)
                alns.append(a)
                s.add(r, res, len(reads), weights[i] if weights is not None else None)
            if fast_order:      # ... and the reference's Kahn order again before consensus / MSA
                import ctypes as C
                spl, fb = C.c_int64(0), C.c_int64(0)
                s.lib.dll.poa_graph_order_stats(s.ab.contents.abg, C.byref(spl), C.byref(fb))
                s.order_stats = (spl.value, fb.value)
                s.lib.dll.poa_graph_set_fast_order(s.ab.contents.abg, 0)
                g = s.ab.contents.abg.contents
                if g.node_n > 2:
                    g.is_topological_sorted = 0
                    s.lib.abpoa_topological_sort(s.ab.contents.abg, s.abpt)
        else:
            alns = s.run_reads(reads, weights=weights)
        s.generate()
        return {
            "order_stats": getattr(s, "order_stats", None),
            "alns": alns,
            "cons": s.consensus(),
            "cov": s.consensus_cov(),
            "msa": s.msa_rows(),
        }


def assert_group_equal(a, b, tag=""):
    from golden_reference import RefGroup, assert_matches_reference
    if isinstance(b, RefGroup):
        return assert_matches_reference(a, b, tag)
    assert len(a["alns"]) == len(b["alns"])
    for i, (x, y) in enumerate(zip(a["alns"], b["alns"])):
        assert x.aligned == y.aligned, f"{tag} read {i}: aligned flag"
        if not x.aligned:
            continue
        assert x.best_score == y.best_score, f"{tag} read {i}: best_score {x.best_score} != {y.best_score}"
        assert x.cigar.shape == y.cigar.shape and np.array_equal(x.cigar, y.cigar), f"{tag} read {i}: graph_cigar differs"
        assert (x.node_s, x.node_e, x.query_s, x.query_e) == (y.node_s, y.node_e, y.query_s, y.query_e), f"{tag} read {i}: ends"
        assert x.cells == y.cells, f"{tag} read {i}: DP cells {x.cells} != {y.cells}"
    assert len(a["cons"]) == len(b["cons"])
    for x, y in zip(a["cons"], b["cons"]):
        assert np.array_equal(x, y), f"{tag}: consensus differs"
    for x, y in zip(a["cov"], b["cov"]):
        assert np.array_equal(x, y), f"{tag}: consensus coverage differs"
    assert len(a["msa"]) == len(b["msa"])
    for x, y in zip(a["msa"], b["msa"]):
        assert np.array_equal(x, y), f"{tag}: RC-MSA differs"


def group_digest(r, m: int = 5):
    """Same shape as the entries of tests/golden/golden.json."""
    import hashlib

    from abpoa_b200.aligner import decode

    def sha(a):
        return hashlib.sha1(a.tobytes()).hexdigest()
    return {
        "alns": [{"aligned": a.aligned, "score": a.best_score, "cells": a.cells, "n_cigar": int(len(a.cigar)), "cigar_sha1": sha(a.cigar),
                  "ends": [a.node_s, a.node_e, a.query_s, a.query_e]} for a in r["alns"]],
        "cons": [decode(c, m) for c in r["cons"]],
        "cov_sha1": [sha(c) for c in r["cov"]],
        "msa_sha1": [sha(x) for x in r["msa"]],
        "msa_len": int(len(r["msa"][0])) if r["msa"] else 0,
    }


def assert_digest_equal(got, want, tag=""):
    assert len(got["alns"]) == len(want["alns"]), tag
    for i, (x, y) in enumerate(zip(got["alns"], want["alns"])):
        assert x == y, f"{tag} read {i}: {x} != {y}"
    for k in ("cons", "cov_sha1", "msa_len", "msa_sha1"):
        assert got[k] == want[k], f"{tag}: {k} differs"
