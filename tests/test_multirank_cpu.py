"""World size 2, 4 and 8 on CPU (torch.distributed gloo through the External transport): the whole
host-side setup path of every algorithm -- tuple generation per rank, redistribute_nonzeros,
block splitting, CSR construction, the 2.5D setup skew -- against the REFERENCE's own code
(oracle/_ref: reference sources compiled with shims, MPI ranks as threads), rank by rank and
bit-exact.  BASELINE.json config 1 (N=2^14, 8 nnz/row, R=16, 1.5D sparse shift, world size 2)
is the first case."""
import pytest

from tests import mp_util as U

CASES_2 = [
    U.case("15d_sparse", 1, 16, 14, 8, name="cfg1_15d_sparse", load="er"),
    U.case("15d_fusion1", 1, 8, 7, 5),
    U.case("15d_fusion2", 2, 8, 7, 5),
    U.case("15d_sparse", 2, 8, 7, 5),
    U.case("25d_sparse_replicate", 2, 8, 7, 5),
    # sizes that do not divide evenly: trailing blocks are padded (ceil-div sizing, common.cpp:20-27)
    U.case("15d_fusion2", 1, 8, 7, 5, n=101),
    U.case("15d_sparse", 1, 8, 7, 5, n=101),
    # rectangular matrices (more columns than rows and the reverse; neither divides evenly)
    U.case("15d_fusion2", 1, 8, 7, 5, n=120, m=75, name="rect_fusion2"),
    U.case("15d_sparse", 2, 8, 7, 5, n=70, m=128, name="rect_sparse"),
    # 650k tuples: the multi-threaded bucketing / counting-sort paths of the setup
    U.case("15d_fusion1", 1, 8, 14, 40, name="big_fusion1"),
    U.case("25d_sparse_replicate", 2, 8, 14, 40, name="big_25d_sparse"),
]
CASES_4 = [
    U.case("15d_fusion1", 2, 8, 7, 5),
    U.case("15d_sparse", 1, 8, 7, 5),
    U.case("25d_dense_replicate", 1, 8, 7, 5),
    U.case("25d_sparse_replicate", 1, 8, 7, 5),
    U.case("15d_fusion1", 2, 8, 7, 5, n=99),
    U.case("25d_dense_replicate", 1, 8, 7, 5, n=99),
    # any initial distribution of the tuples is legal input: all on the last rank / scattered and handed over unsorted
    dict(U.case("15d_fusion2", 2, 8, 7, 5, n=101, m=90, name="deal_last"), deal="last"),
    dict(U.case("15d_sparse", 1, 8, 7, 5, n=101, m=90, name="deal_scatter"), deal="scatter"),
    # 16 x 16 with one nonzero per row on 4 ranks: null blocks and empty CSR blocks
    U.case("15d_fusion1", 1, 4, 4, 1, name="tiny_fusion1"),
    U.case("15d_fusion2", 2, 4, 4, 1, name="tiny_fusion2"),
    U.case("15d_sparse", 4, 4, 4, 1, name="tiny_sparse"),
    U.case("25d_dense_replicate", 1, 4, 4, 1, name="tiny_25d_dense"),
    U.case("25d_sparse_replicate", 1, 4, 4, 1, name="tiny_25d_sparse"),
    U.case("15d_fusion1", 1, 8, 7, 5, n=100, m=61, name="rect_fusion1"),
    U.case("25d_dense_replicate", 1, 8, 7, 5, n=90, m=128, name="rect_25d_dense"),
    U.case("25d_sparse_replicate", 1, 8, 7, 5, n=128, m=77, name="rect_25d_sparse"),
]
# the grid shapes of the 8-GPU runs (BASELINE.json configs 2-5): p=8 with c = 1, 2, 4, 8; 2.5D with s=2, c=2
CASES_8 = [
    U.case("15d_fusion2", 1, 8, 7, 5),
    U.case("15d_fusion1", 4, 8, 7, 5),
    U.case("15d_fusion2", 8, 8, 7, 5),
    U.case("15d_sparse", 2, 8, 7, 5),
    U.case("25d_dense_replicate", 2, 8, 7, 5),
    U.case("25d_sparse_replicate", 2, 8, 7, 5),
]


@pytest.mark.parametrize("nproc,cases", [(2, CASES_2), (4, CASES_4), (8, CASES_8)])
def test_setup_path_matches_reference_rank_by_rank(nproc, cases):
    cases = [dict(c, script=[]) for c in cases]
    got = U.run_cases(nproc, cases, "gloo")
    for c in cases:
        want, src = U.reference_for(dict(c, script=[]), nproc)
        assert want is not None, f"no reference for {c['name']} (p={nproc}): run scripts/make_golden.py"
        U.compare_layout(got[c["name"]], want, c["alg"])
