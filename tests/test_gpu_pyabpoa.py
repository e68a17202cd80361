"""GPU: the pyabpoa-compatible surface (abpoa_b200.aligner.msa_aligner mirrors python/pyabpoa.pyx:93-371) must give
what the reference library gives for the same calls -- the very same driver is run over libabpoa_b200.so and, to
record the stored answers (tests/golden_reference.py), over the reference library (lib=...), so every field of
msa_result is compared."""
import json

import numpy as np
import pytest

from abpoa_b200 import synth
from abpoa_b200.aligner import decode, msa_aligner
from golden_reference import digest

pytestmark = pytest.mark.gpu

EXAMPLE = [   # python/example.py, second example
    "CGTCAATCTATCGAAGCATACGCGGGCAGAGCCGAAGACCTCGGCAATCCA",
    "CCACGTCAATCTATCGAAGCATACGCGGCAGCCGAACTCGACCTCGGCAATCAC",
    "CGTCAATCTATCGAAGCATACGCGGCAGAGCCCGGAAGACCTCGGCAATCAC",
    "CGTCAATGCTAGTCGAAGCAGCTGCGGCAGAGCCGAAGACCTCGGCAATCAC",
    "CGTCAATCTATCGAAGCATTCTACGCGGCAGAGCCGACCTCGGCAATCAC",
    "CGTCAATCTAGAAGCATACGCGGCAAGAGCCGAAGACCTCGGCCAATCAC",
    "CGTCAATCTATCGGTAAAGCATACGCTCTGTAGCCGAAGACCTCGGCAATCAC",
    "CGTCAATCTATCTTCAAGCATACGCGGCAGAGCCGAAGACCTCGGCAATC",
    "CGTCAATGGATCGAGTACGCGGCAGAGCCGAAGACCTCGGCAATCAC",
    "CGTCAATCTAATCGAAGCATACGCGGCAGAGCCGTCTACCTCGGCAATCACGT",
]


FIELDS = ("n_seq", "n_cons", "clu_n_seq", "clu_read_ids", "cons_len", "cons_seq", "cons_cov", "cons_qv", "msa_len", "msa_seq")


def fields(res):
    """Digest of every field of an msa_result."""
    plain = lambda v: json.loads(json.dumps(v, default=lambda o: o.tolist() if hasattr(o, "tolist") else int(o)))
    return {f: digest(plain(getattr(res, f))) for f in FIELDS}


def same(a, b):
    a = fields(a)
    for f in FIELDS:
        assert a[f] == b[f], f


def reference(reference_lib, question, run):
    """The reference's msa_result digests for `run(lib)` (stored; `question` names the call)."""
    return reference_lib.value("pyabpoa", question, lambda lib: [fields(x) for x in run(lib)])


@pytest.mark.parametrize("mode", ["g", "l", "e"])
def test_msa_example(product_lib, reference_lib, mode):
    a = msa_aligner(aln_mode=mode, lib=product_lib).msa(EXAMPLE, out_cons=True, out_msa=True)
    b, = reference(reference_lib, ("example", mode, EXAMPLE), lambda lib: [msa_aligner(aln_mode=mode, lib=lib).msa(EXAMPLE, out_cons=True, out_msa=True)])
    same(a, b)
    if mode == "g":
        assert a.cons_seq[0] == "CGTCAATCTATCGAAGCATACGCGGCAGAGCCGAAGACCTCGGCAATCAC"     # SURVEY 8c
        assert a.msa_len == 75


def test_msa_consensus_only_and_qscores(product_lib, reference_lib):
    reads = [decode(r) for r in synth.make_group(6100, 8, 400, 0.06)]
    rng = np.random.default_rng(3)
    qs = [rng.integers(1, 41, size=len(r)).tolist() for r in reads]
    for kw in (dict(), dict(qscores=qs)):
        a = msa_aligner(lib=product_lib).msa(reads, out_cons=True, out_msa=False, **kw)
        b, = reference(reference_lib, ("consensus_only", reads, kw), lambda lib: [msa_aligner(lib=lib).msa(reads, out_cons=True, out_msa=False, **kw)])
        same(a, b)


def test_incremental_msa_align_add_output(product_lib, reference_lib):
    reads = [decode(r) for r in synth.make_group(6200, 9, 300, 0.05)]

    def run(lib):
        al = msa_aligner(match=3, mismatch=5, gap_open1=5, gap_open2=30, lib=lib)
        al.msa_align(reads[:4], out_cons=True, out_msa=True)
        first = al.msa_output()
        al.msa_add(reads[4:7]).msa_add(reads[7:])
        return first, al.msa_output()
    a, b = run(product_lib), reference(reference_lib, ("incremental", reads), run)
    same(a[0], b[0])
    same(a[1], b[1])


def test_amino_acid_score_matrix(product_lib, reference_lib):
    from abpoa_b200.capi import REPO_ROOT
    mtx = str(REPO_ROOT / "abpoa_b200" / "data" / "BLOSUM62.mtx")
    reads = [decode(r, 27) for r in synth.make_group(6300, 6, 250, 0.10, m=27)]
    a = msa_aligner(is_aa=True, score_matrix=mtx, gap_open2=0, gap_ext2=0, lib=product_lib).msa(reads, True, True)
    b, = reference(reference_lib, ("amino_acid", mtx, reads),
                   lambda lib: [msa_aligner(is_aa=True, score_matrix=mtx, gap_open2=0, gap_ext2=0, lib=lib).msa(reads, True, True)])
    same(a, b)
