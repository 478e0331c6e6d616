"""The compile-time-shape instantiations of the TMA-input kernel (MTG_OPT_V5_STATIC_SHAPE) against the run-time-shape
kernel: bitwise equal coefficients, status and d_free, on every specialised shape, at batch sizes from one tile to a
million trajectories, with the static and the dynamic tile counter, and with non-positive segment times; shapes
without an instantiation route exactly as with the option off."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ON, OFF = 0, -1


def _inputs(N, K, D, B, seed, bad_times=False):
    import torch
    import oracle_lib
    rng = np.random.RandomState(seed)
    pos = rng.uniform(-10, 10, size=(B, K + 1, D))
    dist = np.maximum(np.linalg.norm(np.diff(pos, axis=1), axis=2), 0.2)
    times = dist / 3.0 * 2 * (1.0 + 6.5 * 3.0 / 5.0 * np.exp(-dist / 3.0 * 2))
    if bad_times:  # zero and negative times on either lane's half of the trajectory, first and last segment included
        for b, j, t in [(0, 0, 0.0), (3, K - 1, -1.0), (17, K // 2, 0.0), (B - 1, 1, -0.5), (B // 2, K // 2 - 1, -2.0)]:
            times[b, j] = t
    sd = rng.uniform(-1, 1, size=(B, N // 2 - 1, D))
    ed = rng.uniform(-1, 1, size=(B, N // 2 - 1, D))
    t_d = torch.from_numpy(np.ascontiguousarray(times)).cuda()
    f_d = torch.from_numpy(oracle_lib.waypoint_d_fixed(N, pos, sd, ed)).cuda()
    return t_d, f_d


def _solve(solver, prob, t_d, f_d, static_shape, dyn):
    import torch
    import mav_trajectory_generation_b200 as m
    B = t_d.shape[0]
    solver.set_option(m.capi.OPT_V5_STATIC_SHAPE, static_shape)
    solver.set_option(m.capi.OPT_DYNAMIC_TILES, dyn)
    try:
        st = torch.full((B,), -7, dtype=torch.int32, device="cuda")
        df = torch.full((B, prob.D, prob.n_free), -7.0, dtype=torch.float64, device="cuda")
        out = solver.solve_linear(prob, t_d, f_d, status=st, d_free=df)
        torch.cuda.synchronize()
    finally:
        solver.set_option(m.capi.OPT_V5_STATIC_SHAPE, ON)
        solver.set_option(m.capi.OPT_DYNAMIC_TILES, 0)
    return out, st, df


def _bits_equal(a, b):
    """bitwise equality of float64 tensors; NaN (the coefficients of a trajectory with a non-positive segment time)
    must sit at the same places, its sign and payload are not compared"""
    import torch
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.masked_fill(na, 0.0).view(torch.int64),
                                               b.masked_fill(nb, 0.0).view(torch.int64))


def _v5_kernels(fn):
    """template arguments of every TMA-input kernel launched by fn()"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "twisted_tmem_v5_kernel" in e.name]
    return [re.search(r"twisted_tmem_v5_kernel<([^>]*)>", n).group(1).replace(" ", "") for n in names]


# (N, r, K, D): the specialised shapes (C5 / C3, C2, C4); B: one tile, a batch that is not a whole number of passes of
# the persistent grid (2 or 3 CTAs x 148 SMs x 64 trajectories), and for K = 16 the million of C5
@pytest.mark.parametrize("N,r,K,D,B", [(10, 4, 16, 3, 16), (10, 4, 16, 3, 40000), (10, 4, 16, 3, 1048576),
                                       (10, 4, 8, 3, 16), (10, 4, 8, 3, 40000), (8, 3, 4, 3, 16), (8, 3, 4, 3, 40000)])
@pytest.mark.parametrize("dyn", [1, 2])
def test_static_shape_bitwise_equal_to_runtime_shape(solver, N, r, K, D, B, dyn):
    import mav_trajectory_generation_b200 as m
    prob = m.Problem(N, r, K, D)
    t_d, f_d = _inputs(N, K, D, B, seed=K * 10 + B % 97)
    off = _solve(solver, prob, t_d, f_d, OFF, dyn)
    on = _solve(solver, prob, t_d, f_d, ON, dyn)
    assert bool((off[1] == 0).all())
    assert _bits_equal(on[0], off[0])
    assert _bits_equal(on[2], off[2])
    assert bool((on[1] == off[1]).all())


@pytest.mark.parametrize("N,r,K,D", [(10, 4, 16, 3), (10, 4, 8, 3), (8, 3, 4, 3)])
@pytest.mark.parametrize("dyn", [1, 2])
def test_static_shape_status_bits_with_nonpositive_times(solver, N, r, K, D, dyn):
    import mav_trajectory_generation_b200 as m
    B = 4096
    prob = m.Problem(N, r, K, D)
    t_d, f_d = _inputs(N, K, D, B, seed=7 + K, bad_times=True)
    off = _solve(solver, prob, t_d, f_d, OFF, dyn)
    on = _solve(solver, prob, t_d, f_d, ON, dyn)
    bad = sorted({0, 3, 17, B - 1, B // 2})
    st = off[1].cpu().numpy()
    assert (st[bad] & m.capi.STATUS_BAD_TIME).all() and (np.delete(st, bad) == 0).all()
    assert bool((on[1] == off[1]).all())
    assert _bits_equal(on[0], off[0])
    assert _bits_equal(on[2], off[2])


@pytest.mark.parametrize("N,r,K,D,B,kc", [(10, 4, 16, 3, 4096, 16), (10, 4, 8, 3, 4096, 8), (8, 3, 4, 3, 4096, 4),
                                          (10, 4, 14, 3, 4096, 0), (10, 4, 12, 3, 4096, 0), (10, 4, 16, 1, 4096, 0)])
def test_static_shape_routing(solver, N, r, K, D, B, kc):
    """The option on launches the instantiation for K where one is built, and otherwise the very kernel the option off
    launches; the option off never launches one."""
    import mav_trajectory_generation_b200 as m
    prob = m.Problem(N, r, K, D)
    t_d, f_d = _inputs(N, K, D, B, seed=5)
    res = {}
    for opt in (OFF, ON):
        res[opt] = _v5_kernels(lambda: res.__setitem__("out%d" % opt, _solve(solver, prob, t_d, f_d, opt, 0)))
    assert len(res[OFF]) == 1 and len(res[ON]) == 1, res
    assert res[OFF][0].split(",")[-1] == "0"
    if kc:
        assert res[ON][0].split(",")[-1] == str(kc)
        assert res[ON][0].split(",")[:-1] == res[OFF][0].split(",")[:-1]
    else:
        assert res[ON] == res[OFF]
    a, b = res["out%d" % OFF], res["out%d" % ON]
    assert _bits_equal(a[0], b[0]) and _bits_equal(a[2], b[2]) and bool((a[1] == b[1]).all())
