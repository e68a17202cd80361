"""What the unmodified reference computes, stored as digests in tests/golden/reference.json.

The parity tests compare the product with the reference (abPOA v1.5.6, AVX2 build) on the same inputs.  The
reference is not part of this repository, so its answers are stored: every answer is filed under a digest of
the question (kind of call, configuration, reads, options) and kept as digests of what the tests compare
(per-read scores, graph-CIGARs, end points, DP cells, consensus, coverage, RC-MSA).  The `reference_lib`
fixture hands the tests a `GoldenReference`; the product's results are digested the same way and compared
field by field.

Regenerating (after a change of the inputs of a test): build the reference into oracle/_ref/ (oracle/Makefile)
and run the whole suite with ABPOA_REFERENCE_RECORD=<file>.  Every question is then answered by the live
reference, the comparisons run against those answers, and the answers of the session are written to <file>,
which replaces tests/golden/reference.json.
"""
from __future__ import annotations

import hashlib
import json
import os
from pathlib import Path

import numpy as np
import pytest

from abpoa_b200.capi import REPO_ROOT

GOLDEN_FILE = Path(__file__).resolve().parent / "golden" / "reference.json"
REFERENCE_LIB = REPO_ROOT / "oracle" / "_ref" / "libabpoa_ref.so"     # built by oracle/Makefile, only for recording
HASH_HEX = 10
GROUP_FIELDS = ("n", "unaligned", "cells", "aln", "bat", "cons", "cov", "msa")     # stored as a list in this order


def _feed(h, x):
    if isinstance(x, np.ndarray):
        x = np.ascontiguousarray(x)
        h.update(f"A{x.dtype.str}{x.shape}".encode())
        h.update(x.tobytes())
    elif isinstance(x, dict):
        h.update(f"D{len(x)}".encode())
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif isinstance(x, (list, tuple)):
        h.update(f"L{len(x)}".encode())
        for y in x:
            _feed(h, y)
    else:
        if isinstance(x, str) and x.startswith(str(REPO_ROOT)):       # paths of data files inside the tree
            x = os.path.relpath(x, REPO_ROOT)
        h.update(f"S{x!r}".encode())


def digest(*parts) -> str:
    h = hashlib.sha1()
    for p in parts:
        _feed(h, p)
    return h.hexdigest()[:HASH_HEX]


def arrays_digest(arrays) -> str:
    """Digest of a list of integer arrays (consensus, coverage, MSA rows), independent of their integer type."""
    return digest([np.asarray(a).astype(np.int64) for a in arrays])


def group_record(r) -> dict:
    """Digest of one progressive MSA (the dict returned by helpers.run_group).

    aln:   per read the aligned flag, best score, every graph-CIGAR word, end points and DP cells;
    bat:   per aligned read the best score, CIGAR length and FNV-1a hash of the CIGAR words (what the batch engine
           reports per read);
    cells: DP cells of the whole group; cons / cov / msa: consensus, its coverage and the RC-MSA rows."""
    from abpoa_b200.batch import fnv1a_words
    alns = r["alns"]
    return {
        "n": len(alns),
        "unaligned": [i for i, a in enumerate(alns) if not a.aligned],
        "cells": int(sum(a.cells for a in alns)),
        "aln": digest([(bool(a.aligned), int(a.best_score), np.asarray(a.cigar, dtype=np.uint64), [int(a.node_s), int(a.node_e), int(a.query_s), int(a.query_e)],
                        int(a.cells)) if a.aligned else (False,) for a in alns]),
        "bat": digest([(i, int(a.best_score), len(a.cigar), fnv1a_words(a.cigar)) for i, a in enumerate(alns) if a.aligned]),
        "cons": arrays_digest(r["cons"]), "cov": arrays_digest(r["cov"]), "msa": arrays_digest(r["msa"]),
    }


class GoldenReference:
    """Stands in for the reference library: answers questions from the stored digests, or, when recording,
    from the live reference (and stores the answers)."""

    def __init__(self, record_to: str | None = None):
        self.record_to = record_to
        self.live = None
        self.answers = {}
        if record_to:
            from abpoa_b200 import capi
            if not REFERENCE_LIB.exists():
                raise RuntimeError(f"recording needs the reference library {REFERENCE_LIB} (oracle/Makefile)")
            self.live = capi.load_library(REFERENCE_LIB)
        self.stored = json.loads(GOLDEN_FILE.read_text()) if GOLDEN_FILE.exists() else {}

    def value(self, kind: str, question, compute):
        """The reference's answer to `question` (any nesting of dicts, lists, scalars and arrays); `compute(lib)`
        asks the live reference and returns a JSON-able answer."""
        key = f"{kind}:{digest(kind, question)}"
        if key in self.answers:
            return self.answers[key]
        if self.live is not None:
            ans = json.loads(json.dumps(compute(self.live)))
        elif key in self.stored:
            ans = self.stored[key]
        else:
            pytest.fail(f"no stored reference answer for {key} (the inputs of this test changed?): regenerate "
                        f"tests/golden/reference.json as described in tests/golden_reference.py")
        self.answers[key] = ans
        return ans

    def group(self, cfg, reads, want_msa=True, weights=None) -> "RefGroup":
        from helpers import run_group
        cfg = dict(cfg.__dict__, out_msa=want_msa)
        question = (cfg, list(reads), weights if weights is None else list(weights))
        rec = self.value("group", question, lambda lib: _pack(group_record(run_group(lib, _config(cfg), reads, want_msa, weights=weights))))
        return RefGroup(zip(GROUP_FIELDS, rec))

    def groups(self, cfg, groups, want_msa=False, procs=4) -> list["RefGroup"]:
        """Many groups, answered by parallel reference processes when recording (the reference is single-threaded
        and, at 10 kbp, page-fault bound: ~15 s per 50-read group)."""
        cfgd = dict(cfg.__dict__, out_msa=want_msa)
        todo = [g for g in groups if self.live is not None and f"group:{digest('group', (cfgd, list(g), None))}" not in self.answers]
        if todo:
            import multiprocessing as mp
            with mp.get_context("spawn").Pool(min(procs, len(todo))) as pool:
                recs = pool.map(_group_worker, [(cfgd, g, want_msa) for g in todo])
            for g, rec in zip(todo, recs):
                self.answers[f"group:{digest('group', (cfgd, list(g), None))}"] = json.loads(json.dumps(_pack(rec)))
        return [self.group(cfg, g, want_msa) for g in groups]

    def save(self):
        if self.record_to:
            Path(self.record_to).write_text(json.dumps(dict(sorted(self.answers.items())), separators=(",", ":")) + "\n")


def _pack(rec: dict) -> list:
    return [rec[f] for f in GROUP_FIELDS]


def _config(d):
    from abpoa_b200.aligner import PoaConfig
    return PoaConfig(**d)


def _group_worker(args):
    from helpers import run_group
    from abpoa_b200 import capi
    cfgd, reads, want_msa = args
    return group_record(run_group(capi.load_library(REFERENCE_LIB), _config(cfgd), reads, want_msa))


class RefGroup(dict):
    """The stored digest of one group (see group_record)."""


def assert_matches_reference(got, ref: RefGroup, tag=""):
    """A progressive MSA of the product (helpers.run_group) against the reference's stored digest."""
    g = group_record(got)
    assert g["n"] == ref["n"], f"{tag}: {g['n']} reads, reference {ref['n']}"
    assert g["unaligned"] == ref["unaligned"], f"{tag}: reads without alignment {g['unaligned']} vs {ref['unaligned']}"
    assert g["aln"] == ref["aln"], f"{tag}: per-read score / graph-CIGAR / end points / DP cells differ (scores {[a.best_score for a in got['alns']]})"
    assert g["cells"] == ref["cells"], f"{tag}: DP cells {g['cells']} != {ref['cells']}"
    assert g["cons"] == ref["cons"], f"{tag}: consensus differs"
    assert g["cov"] == ref["cov"], f"{tag}: consensus coverage differs"
    assert g["msa"] == ref["msa"], f"{tag}: RC-MSA differs"


def assert_batch_matches_reference(r, ref: RefGroup, tag="", cells=True, msa=True):
    """One group of the batch engine (batch.GroupResult with per-read records) against the reference's digest:
    DP cells, per aligned read the best score, CIGAR length and CIGAR hash, consensus, coverage (and RC-MSA)."""
    if cells:
        assert r.dp_cells == ref["cells"], f"{tag}: cells {r.dp_cells} != {ref['cells']}"
    aligned = [i for i in range(ref["n"]) if i not in ref["unaligned"]]
    got = digest([(i, int(r.read_best_score[i]), int(r.read_n_cigar[i]), int(r.read_cigar_hash[i])) for i in aligned])
    assert got == ref["bat"], f"{tag}: per-read score / CIGAR length / CIGAR hash differ (scores {[int(r.read_best_score[i]) for i in aligned]})"
    assert arrays_digest(r.cons) == ref["cons"], f"{tag}: consensus"
    assert arrays_digest(r.cov) == ref["cov"], f"{tag}: coverage"
    if msa:
        assert arrays_digest(r.msa) == ref["msa"], f"{tag}: msa"
