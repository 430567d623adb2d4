"""The carry kernel of the time-sharded passes (behind moihgp_cuda_fsn_carry_dev and moihgp_cuda_carry_in_dev): the limit
of 64 time blocks, and the carries across 64 blocks against the host algebra of parallel.py (forward_carry_in,
backward_carry_in, carry_in_from_block_ends)."""
import numpy as np
import pytest

from conftest import rel_err

MAX_BLOCKS = 64


def _model(kernel, p, L):
    from multioutputihgp_b200 import MOIHGPSequences
    from oracle.gen_golden import make_params
    m = MOIHGPSequences(0.1, p, L, kernel, True)
    m.update(make_params(np.random.default_rng(3), p, L, kernel))
    return m


@pytest.mark.gpu
def test_more_than_64_blocks_are_refused(cuda_lib):
    import torch
    m = _model("Matern32", 8, 4)
    N, L, d, G = 2, 4, m.igp_dim, MAX_BLOCKS + 1
    f64 = dict(dtype=torch.float64, device=torch.device("cuda:0"))
    lengths = [256] * G
    out = torch.zeros((N, L, d), **f64)
    for direction, w in ((0, d + 1), (1, d)):
        with pytest.raises(RuntimeError, match="G <= 64 time blocks"):
            m.fsn_carry_device(direction, torch.zeros((G, N, L, w), **f64), lengths, 0, out)
    with pytest.raises(RuntimeError, match="G <= 64 time blocks"):
        m.carry_in_device(torch.zeros((G, N, L, 4, d), **f64), lengths, 1, out, torch.zeros((N, L, 3, d), **f64))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["Matern32", "Matern52"])
@pytest.mark.parametrize("mode", [1, 0])
def test_carries_of_64_blocks_match_the_host_algebra(cuda_lib, kernel, mode):
    """64 blocks of random records; lengths log-uniform up to 10^6 (short ones, whose carries reach far, and long ones),
    with a run of equal lengths.  Forward and backward filter + smoother carries in both smoother modes, and the objective's
    carry-in, for the first, second, a middle and the last block."""
    import torch
    from multioutputihgp_b200.parallel import backward_carry_in, carry_in_from_block_ends, forward_carry_in
    m = _model(kernel, 8, 4)
    N, L, d, G = 2, 4, m.igp_dim, MAX_BLOCKS
    rng = np.random.default_rng(41 + mode)
    lengths = [int(v) for v in np.round(10 ** rng.uniform(0, 6, G))]
    lengths[10:20] = [lengths[9]] * 10
    g1, g2 = rng.standard_normal((G, N, L, d + 1)), rng.standard_normal((G, N, L, d))
    ends, x0, dx0 = rng.standard_normal((G, N, L, 4, d)), rng.standard_normal((N, L, d)), rng.standard_normal((N, L, 3, d))
    dev = torch.device("cuda:0")
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    g1d, g2d, endsd, x0d, dx0d = (to_dev(a) for a in (g1, g2, ends, x0, dx0))
    for rank in (0, 1, 37, G - 1):
        xin, bend, cx, cdx = (torch.zeros(s, dtype=torch.float64, device=dev) for s in ((N, L, d), (N, L, d), (N, L, d), (N, L, 3, d)))
        uaf = torch.full((N, L), 7.0, dtype=torch.float64, device=dev)
        bend.fill_(7.0)
        m.fsn_carry_device(0, g1d, lengths, rank, xin, mode, x0=x0d, u_after=uaf)
        m.fsn_carry_device(1, g2d, lengths, rank, bend, mode)
        m.carry_in_device(endsd, lengths, rank, cx, cdx, x0=x0d, dx0=dx0d)
        torch.cuda.synchronize()
        xh = forward_carry_in(m.block_transition, lengths, list(g1[..., :d]), x0, rank)
        assert rel_err(xin.cpu().numpy(), xh) < 1e-13, rank
        bh = backward_carry_in(lambda n_: m.smoother_power(n_, mode), lengths, list(g2), rank)
        if bh is None:                                       # the last block: nothing comes from the right
            assert (uaf.cpu().numpy() == 7.0).all() and (bend.cpu().numpy() == 7.0).all(), rank
        else:
            assert np.array_equal(uaf.cpu().numpy(), g1[rank + 1][..., d]), rank
            bd = bend.cpu().numpy()                          # literal mode: a latent with rho(G) > 1 overflows on both sides
            assert np.array_equal(np.isfinite(bd), np.isfinite(bh)), rank
            for l in range(L):
                if np.isfinite(bh[:, l]).all() and np.max(np.abs(bh[:, l])) < 1e100:
                    assert rel_err(bd[:, l], bh[:, l]) < 1e-13, (rank, l)
        for n in range(N):
            ch, cdh = carry_in_from_block_ends(m.block_transition, lengths, ends[:, n, :, 0], ends[:, n, :, 1:], x0[n], dx0[n], rank)
            assert rel_err(cx[n].cpu().numpy(), ch) < 1e-13 and rel_err(cdx[n].cpu().numpy(), cdh) < 1e-13, (rank, n)
