"""Drop-in boundary against the REFERENCE's public interface (CPU):

* struct layout: a probe compiled against include/abpoa.h must print the same sizeof / offsetof for every public struct and
  the same values for every constant as the same probe compiled against the reference's abpoa.h (its output is stored in
  tests/golden/reference_abi.txt);
* every function of abpoa.h that the reference's example programs (example.c, sub_example.c, incre_example.c) call -- the
  lists are stored in tests/golden/reference_example_api.json -- is declared by OUR header and exported by
  libabpoa_b200.so: a program taking the address of each one compiles and links (running the calls needs a GPU; on a GPU
  box the library's own tests cover them)."""
import json
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = Path(__file__).resolve().parent / "golden"
LIBDIR = ROOT / "abpoa_b200" / "lib"

PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include "abpoa.h"
#define S(t) printf("sizeof " #t " %zu\n", sizeof(t))
#define O(t, f) printf("offsetof " #t "." #f " %zu\n", offsetof(t, f))
#define K(c) printf(#c " %ld\n", (long)(c))
int main(void) {
    S(abpoa_res_t); O(abpoa_res_t, n_cigar); O(abpoa_res_t, graph_cigar); O(abpoa_res_t, node_s); O(abpoa_res_t, query_e); O(abpoa_res_t, n_matched_bases); O(abpoa_res_t, best_score);
    S(abpoa_para_t); O(abpoa_para_t, m); O(abpoa_para_t, mat); O(abpoa_para_t, mat_fn); O(abpoa_para_t, use_score_matrix); O(abpoa_para_t, match); O(abpoa_para_t, max_mat);
    O(abpoa_para_t, mismatch); O(abpoa_para_t, min_mis); O(abpoa_para_t, gap_open1); O(abpoa_para_t, gap_ext2); O(abpoa_para_t, inf_min); O(abpoa_para_t, k); O(abpoa_para_t, w);
    O(abpoa_para_t, min_w); O(abpoa_para_t, wb); O(abpoa_para_t, wf); O(abpoa_para_t, zdrop); O(abpoa_para_t, end_bonus); O(abpoa_para_t, incr_fn); O(abpoa_para_t, out_pog);
    O(abpoa_para_t, align_mode); O(abpoa_para_t, gap_mode); O(abpoa_para_t, max_n_cons); O(abpoa_para_t, cons_algrm); O(abpoa_para_t, min_freq); O(abpoa_para_t, verbose); O(abpoa_para_t, batch_index);
    S(abpoa_node_t); O(abpoa_node_t, node_id); O(abpoa_node_t, in_edge_n); O(abpoa_node_t, in_id); O(abpoa_node_t, out_edge_n); O(abpoa_node_t, out_id); O(abpoa_node_t, in_edge_weight);
    O(abpoa_node_t, out_edge_weight); O(abpoa_node_t, read_weight); O(abpoa_node_t, n_read); O(abpoa_node_t, read_ids); O(abpoa_node_t, aligned_node_n); O(abpoa_node_t, aligned_node_id);
    O(abpoa_node_t, n_span_read); O(abpoa_node_t, base);
    S(abpoa_graph_t); O(abpoa_graph_t, node); O(abpoa_graph_t, node_n); O(abpoa_graph_t, index_to_node_id); O(abpoa_graph_t, node_id_to_index); O(abpoa_graph_t, node_id_to_max_pos_left);
    O(abpoa_graph_t, node_id_to_max_remain); O(abpoa_graph_t, node_id_to_msa_rank);
    S(abpoa_cons_t); O(abpoa_cons_t, n_cons); O(abpoa_cons_t, n_seq); O(abpoa_cons_t, msa_len); O(abpoa_cons_t, clu_n_seq); O(abpoa_cons_t, clu_read_ids); O(abpoa_cons_t, cons_len);
    O(abpoa_cons_t, cons_node_ids); O(abpoa_cons_t, cons_base); O(abpoa_cons_t, msa_base); O(abpoa_cons_t, cons_cov); O(abpoa_cons_t, cons_phred_score);
    S(abpoa_str_t); S(abpoa_seq_t); O(abpoa_seq_t, n_seq); O(abpoa_seq_t, seq); O(abpoa_seq_t, name); O(abpoa_seq_t, comment); O(abpoa_seq_t, qual); O(abpoa_seq_t, is_rc);
    S(abpoa_simd_matrix_t); O(abpoa_simd_matrix_t, s_mem); O(abpoa_simd_matrix_t, s_msize); O(abpoa_simd_matrix_t, dp_beg); O(abpoa_simd_matrix_t, dp_end_sn); O(abpoa_simd_matrix_t, rang_m);
    S(abpoa_t); O(abpoa_t, abg); O(abpoa_t, abs); O(abpoa_t, abm); O(abpoa_t, abc);
    K(ABPOA_GLOBAL_MODE); K(ABPOA_LOCAL_MODE); K(ABPOA_EXTEND_MODE); K(ABPOA_LINEAR_GAP); K(ABPOA_AFFINE_GAP); K(ABPOA_CONVEX_GAP);
    K(ABPOA_CMATCH); K(ABPOA_CINS); K(ABPOA_CDEL); K(ABPOA_CDIFF); K(ABPOA_CSOFT_CLIP); K(ABPOA_CHARD_CLIP);
    K(ABPOA_SRC_NODE_ID); K(ABPOA_SINK_NODE_ID); K(ABPOA_OUT_CONS); K(ABPOA_OUT_MSA); K(ABPOA_OUT_CONS_MSA); K(ABPOA_OUT_GFA); K(ABPOA_OUT_CONS_GFA); K(ABPOA_OUT_CONS_FQ);
    K(ABPOA_HB); K(ABPOA_MF);
    return 0;
}
'''


def probe(tmp_path, tag, include_dirs):
    src = tmp_path / f"probe_{tag}.c"
    src.write_text(PROBE)
    exe = tmp_path / f"probe_{tag}"
    subprocess.run(["gcc", "-O0", "-w", *[f"-I{d}" for d in include_dirs], "-DUSE_SIMDE", "-DSIMDE_ENABLE_NATIVE_ALIASES", "-mavx2", "-o", str(exe), str(src)], check=True)
    return subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout


def test_public_structs_match_the_reference_header(tmp_path):
    ours = probe(tmp_path, "ours", [ROOT / "include"])
    theirs = (GOLDEN / "reference_abi.txt").read_text()
    assert ours == theirs, "\n".join(f"{a}   |   {b}" for a, b in zip(ours.splitlines(), theirs.splitlines()) if a != b)


@pytest.mark.parametrize("prog", ["example.c", "sub_example.c", "incre_example.c"])
def test_reference_example_api_links_against_this_library(tmp_path, prog):
    if not (LIBDIR / "libabpoa_b200.so").exists():
        pytest.skip("library not built")
    fns = json.loads((GOLDEN / "reference_example_api.json").read_text())[prog]
    assert fns
    src = tmp_path / ("uses_" + prog)
    src.write_text('#include <stdio.h>\n#include "abpoa.h"\nint main(void) {\n'
                   + "".join(f'    printf("%p\\n", (void *)&{f});\n' for f in fns) + "    return 0;\n}\n")
    exe = tmp_path / src.stem
    r = subprocess.run(["gcc", "-O1", "-Wall", "-Werror=implicit-function-declaration", f"-I{ROOT / 'include'}", "-o", str(exe), str(src),
                        f"-L{LIBDIR}", "-labpoa_b200", f"-Wl,-rpath,{LIBDIR}", "-Wl,--no-undefined", "-lm", "-lz", "-lpthread"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
