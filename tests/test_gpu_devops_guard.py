"""The INT8 accuracy guard of the primitive contraction (DevOps.contract -> DeviceEris.guarded): a product whose
worst-case INT8 error bound exceeds int8_tol is repeated on the FP64 DMMA kernels, one that accumulates into its output
(beta != 0) is refused.  The container holds vvvv / ovvv_p as digit planes only: a primitive contraction names its
operands, so its repeat does not need the FP64 integral layouts that a plan's repeat reads."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ecw(built_lib):
    import ecw_cc_b200
    return ecw_cc_b200


def test_primitive_contraction_guard(ecw):
    import torch
    # int8_min_flops=0: the guard reads the bound of every contraction (a negative threshold routes every GEMM to
    # INT8 but skips the guard of the primitive ops); a 1024^3 product takes the INT8 route (ecw_plan_dump_contract)
    de = ecw.DeviceEris.synthetic(8, 16, gemm="int8", int8_digits=6, int8_min_flops=0)
    ops = de.ops
    assert not de.can_dmma()
    rng = np.random.default_rng(11)
    n = 1024
    a_small, b_small = 1e-3 * rng.standard_normal((n, n)), 1e-3 * rng.standard_normal((n, n))
    ops.contract("ij,jk->ik", ops.to_dev(a_small), ops.to_dev(b_small))
    assert de.guard_trips == 0 and 0.0 < de.last_bound <= de.int8_tol and de.max_bound == de.last_bound

    A, B = 100.0 * rng.standard_normal((n, n)), 100.0 * rng.standard_normal((n, n))
    dA, dB = ops.to_dev(A), ops.to_dev(B)
    got = ops.contract("ij,jk->ik", dA, dB).cpu().numpy()
    assert de.guard_trips == 1 and de.last_bound > de.int8_tol
    assert de.max_bound < de.int8_tol                          # a tripped bound is not recorded as the largest seen
    ref = torch.einsum("ij,jk->ik", dA, dB).cpu().numpy()     # FP64 (cuBLAS)
    scale = np.abs(ref).max()
    assert scale > 1e5 and np.abs(got - ref).max() < 1e-13 * scale

    C0 = rng.standard_normal((n, n))
    dC = ops.to_dev(C0)
    with pytest.raises(ecw.EcwError, match="accumulating"):
        ops.contract("ij,jk->ik", dA, dB, out=dC, beta=1.0)
    assert de.guard_trips == 2
