"""-m gpu: the two paths of TT rounding.  With rank caps on every bond and full-rank left unfoldings both sweeps are
enqueued with one synchronisation (speculative); otherwise, and whenever the device flags the speculation, the
host-driven sweeps run.  Both must give the same answer."""
import numpy as np
import pytest
import torch

from gpu_util import ranks_of, relerr64
from oracle import cases

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-10), (np.float32, 2e-6)])
def test_speculative_and_host_driven_rounding_agree(dtype, tol):
    from tntorch_b200 import ops

    cores = cases.random_tt((6, 7, 5, 8, 6), 6, seed=31, dtype=dtype)
    dense = cases.tt_full([c.astype(np.float64) for c in cores])
    dev = [torch.as_tensor(c).cuda() for c in cores]
    rmax = [3, 4, 2, 3]
    _, info = ops.tt_round_batch([dev], rmax=rmax, return_info=True)
    assert info["speculative"] == [1]  # the input takes the speculative path
    spec = ops.tt_round(dev, rmax=rmax)
    host = ops.tt_round(dev, rmax=rmax, speculate=False)
    assert ranks_of(spec) == ranks_of(host) == [1, 3, 4, 2, 3, 1]
    e_spec, e_host = relerr64(dense, spec), relerr64(dense, host)
    assert 0 < e_host < 1
    assert abs(e_spec - e_host) <= tol, (e_spec, e_host)


def test_round_batch_with_a_tensor_that_needs_the_host_driven_path():
    """a + a has rank-deficient left unfoldings: the Cholesky-QR of the speculative phase A flags it and that tensor
    is rounded again host-driven; the others keep their speculative result.  Every result equals the single call."""
    from tntorch_b200 import ops

    shape, rmax = (8, 9, 7, 8), 4
    trains = [[torch.as_tensor(c).cuda() for c in cases.random_tt(shape, 6, seed=40 + b)] for b in range(4)]
    a = [torch.as_tensor(c).cuda() for c in cases.random_tt(shape, 3, seed=50)]
    trains[2] = [c.clone() for c in ops.tt_sum([a, a])]
    assert [c.shape for c in trains[2]] == [c.shape for c in trains[0]]
    out, info = ops.tt_round_batch(trains, rmax=rmax, return_info=True)
    assert info["speculative"] == [1, 1, 0, 1]
    for b in range(4):
        dense = cases.tt_full([c.cpu().numpy() for c in trains[b]])
        ref = ops.tt_round(trains[b], rmax=rmax)
        assert ranks_of(out[b]) == ranks_of(ref)
        assert abs(relerr64(dense, out[b]) - relerr64(dense, ref)) <= 1e-10
