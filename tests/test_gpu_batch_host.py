"""Host side of the batch verbs: the checkpoint format of each Sigma layout, and the batch-size limit.

A checkpoint holds the arrays exactly as the engine keeps them.  Its length per filter is part of the saved format:
tile layout (n = 20) Sigma 1,136 doubles (Sigma and state in one block) and state 44; staircase layout (other n <= 64)
sym_sig_stride(N) and sym_st_stride(N); wide layout (64 < n <= 1,024) N * ld and ld, with ld = N rounded up to 16."""
import numpy as np
import pytest

from _batch import stair_strides

pytestmark = pytest.mark.gpu


def _expected(n):
    """(Sigma doubles, state doubles, state stride in memory) per filter."""
    N = 3 + 2 * n
    if n == 20:
        return 1136, 44, 1136
    if n <= 64:
        sig, st = stair_strides(N)
        return sig, st, st
    ld = (N + 15) & ~15
    return N * ld, ld, ld


@pytest.mark.parametrize("n", [20, 33, 100])
def test_checkpoint_format_per_layout(gpu_pkg, n):
    B, N = 5, 3 + 2 * n
    rng = np.random.default_rng(n)
    bt = gpu_pkg.EKFBatch(B, n)
    for _ in range(2):
        bt.step_known(rng.uniform(-0.05, 0.05, (B, 2)), rng.uniform(-2, 2, (B, 2 * n)),
                      (rng.random((B, n)) < 0.4).astype(np.uint8))
    bt.sync()
    sig_len, st_len, st_stride = _expected(n)
    ck = bt.checkpoint()
    assert ck["sigma_packed"].size == B * sig_len
    assert ck["state"].size == B * st_len
    assert bt.device_pointers()[1::2] == (sig_len, st_stride)
    # the state array starts each filter's block with its state vector
    states = bt.states()
    assert np.array_equal(ck["state"].reshape(B, st_len)[:, :N], states)
    if n > 64:  # the wide layout's Sigma is dense rows of stride ld
        dense = ck["sigma_packed"].reshape(B, N, st_len)
        for b in (0, B - 1):
            assert np.array_equal(dense[b, :, :N], bt.sigma(b))
    # and it restores to the same batch
    other = gpu_pkg.EKFBatch(B, n)
    other.restore(ck)
    assert np.array_equal(other.states(), states)
    for b in (0, B - 1):
        assert np.array_equal(other.sigma(b), bt.sigma(b))
    again = other.checkpoint()
    for k in ("sigma_packed", "state", "init_flag", "known"):
        assert np.array_equal(again[k], ck[k]), k


def test_batch_too_large_for_one_launch_is_invalid(gpu_pkg):
    """Refused as an invalid shape before anything is allocated (not as a failed allocation)."""
    with pytest.raises(gpu_pkg.EkfError) as e:
        gpu_pkg.EKFBatch(2**31, 20)
    assert e.value.code == -1
