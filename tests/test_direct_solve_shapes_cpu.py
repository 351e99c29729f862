"""Host-only check (diffopt_b200_sparse_analyze, no GPU) that the arrowhead generators of test_direct_solve_variants_gpu.py
give the multifrontal analysis the fronts they were built for, before any GPU time is spent on them: exactly D dense
vertices, eliminated last in one root front of order D whose shared-memory size picks the intended factor kernel, and no
front larger than a leaf (<= 32 pivots) over those D rows plus its two chain neighbours."""
import pytest

import diffopt_b200
from test_direct_solve_variants_gpu import MF_CASES, MF_LEAF, MF_ROOT_CLASS, arrowhead, dense_vertex_count, mf_factor_class


@pytest.mark.parametrize("D", [c[0] for c in MF_CASES])
@pytest.mark.parametrize("trans", [False, True])
def test_arrowhead_front_orders(D, trans):
    lsq = diffopt_b200.submodule("lsqr")
    K = arrowhead(D)
    assert dense_vertex_count(K) == D
    assert mf_factor_class(D) == MF_ROOT_CLASS[D]
    st = lsq.sparse_analyze(K, trans=trans)
    assert D <= st["max_front"] <= D + MF_LEAF + 2, st
    assert st["levels"] >= 3, st   # leaves, chain separators, root
