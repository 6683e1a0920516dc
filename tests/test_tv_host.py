"""not-gpu: the TV prox restatement (tests/tv_reference.py) solves the problem it claims to, follows deepinv's restart /
warm-start rules, and the C ABI of the TV prox rejects bad arguments on the host before any CUDA call."""
import ctypes

import pytest
import torch

import tv_reference as TV


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


@pytest.mark.parametrize("shape", [(2, 3, 7, 5), (1, 3, 17, 23), (1, 3, 1, 9), (1, 3, 11, 1), (1, 3, 1, 1)])
def test_nabla_adjoint_is_the_adjoint(shape):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(shape, generator=g, dtype=torch.float64)
    u = torch.randn(shape + (2,), generator=g, dtype=torch.float64)
    lhs, rhs = float((TV.nabla(x) * u).sum()), float((x * TV.nabla_adjoint(u)).sum())
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs))


def test_chambolle_pock_closes_the_primal_dual_gap():
    """crit = 0, fp64, ths = 0.1 on a 3 x 17 x 23 image: the gap of 1/2 ||x - y||^2 + ths TV(x) against the dual point u2 projected
    onto ||u_p|| <= ths falls to <= 1e-8 relative (9.7e-10 measured after 2 000 iterations)."""
    y = torch.rand((1, 3, 17, 23), generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    den = TV.TVDenoiser(n_it_max=2000, crit=0.0)
    x = den.forward(y, 0.1)
    assert den.last_iterations.tolist() == [2000]
    gap = TV.primal_dual_gap(y, x, den.u2, 0.1)
    assert 0 <= gap <= 1e-8, gap


def test_restart_and_warm_start():
    g = torch.Generator().manual_seed(1)
    y = torch.rand((2, 3, 9, 13), generator=g, dtype=torch.float64)
    one = TV.TVDenoiser(n_it_max=10, crit=0.0)
    ref = one.forward(y, 0.05)
    two = TV.TVDenoiser(n_it_max=5, crit=0.0)
    two.forward(y, 0.05)
    x = two.forward(y, 0.05)  # warm start: the same 10 iterations
    assert torch.equal(x, ref) and torch.equal(two.u2, one.u2)
    two.reset()  # restart: x2 = y, u2 = 0 again
    assert torch.equal(two.forward(y, 0.05), TV.TVDenoiser(n_it_max=5, crit=0.0).forward(y, 0.05))
    two.restart = True
    assert torch.equal(two.forward(y, 0.05), TV.TVDenoiser(n_it_max=5, crit=0.0).forward(y, 0.05))
    y1 = y[:1].clone()  # a shape change restarts
    assert torch.equal(two.forward(y1, 0.05), TV.TVDenoiser(n_it_max=5, crit=0.0).forward(y1, 0.05))


def test_huge_crit_stops_after_three_iterations():
    y = torch.rand((3, 3, 8, 8), generator=torch.Generator().manual_seed(2))
    den = TV.TVDenoiser(crit=1e30)
    den.forward(y, 0.1)
    assert den.last_iterations.tolist() == [3, 3, 3]


def test_constant_chain_stops_alone():
    """Per-chain stopping: a constant image is a fixed point (x_prev == x2 from the first iteration) and stops at 3 while a noisy
    chain next to it goes on and stops exactly where it stops alone, with the same state."""
    g = torch.Generator().manual_seed(3)
    noisy = torch.rand((1, 3, 12, 10), generator=g)
    y = torch.cat([torch.full_like(noisy, 0.25), noisy])
    den, alone = TV.TVDenoiser(n_it_max=300), TV.TVDenoiser(n_it_max=300)
    x = den.forward(y, 0.1)
    xa = alone.forward(noisy, 0.1)
    assert den.last_iterations[0] == 3 and den.last_iterations[1] == alone.last_iterations[0] > 3
    assert torch.equal(x[1:], xa) and torch.allclose(x[0], y[0], rtol=0, atol=1e-6)


def test_tv_struct_and_sizes(built):
    L = built._lib
    assert ctypes.sizeof(L.TVParams) == 24
    assert L.lib().psgla_struct_size(5) == ctypes.sizeof(L.TVParams)
    lib = L.lib()
    s = L.ImgShape(2, 3, 5, 7)
    assert lib.psgla_tv_state_bytes(s) == 2 * 3 * 5 * 7 * 12
    assert lib.psgla_tv_workspace_bytes(s) >= 2 * 3 * 5 * 7 * 12
    for bad in (L.ImgShape(0, 3, 5, 7), L.ImgShape(1, 1, 5, 7), L.ImgShape(1, 3, 0, 7), L.ImgShape(1, 3, 5, 0)):
        assert lib.psgla_tv_state_bytes(bad) == 0 and lib.psgla_tv_workspace_bytes(bad) == 0


def test_tv_argument_errors_without_gpu(built):
    """psgla_tv_prox_post rejects each bad argument on the host before any CUDA call (fake pointers are never dereferenced)."""
    L = built._lib
    lib = L.lib()
    fake = 0x1000
    shape = L.ImgShape(1, 3, 8, 8)
    st, ws = lib.psgla_tv_state_bytes(shape), lib.psgla_tv_workspace_bytes(shape)
    post = L.PostParams(1.0, 0.0, 0.0, 1.0)

    def call(prm=None, shape=shape, y=fake, state=fake, st=st, ws_ptr=fake, ws=ws, post=post, out=fake, mean=None, mean2=None):
        prm = L.TVParams(0.1, 0.01, 1.99, 1e-5, 1000, 1) if prm is None else prm
        return lib.psgla_tv_prox_post(ctypes.byref(prm) if prm != "null" else None, shape, y, state, st, ws_ptr, ws,
                                      ctypes.byref(post) if post is not None else None, out, None, mean, mean2, None, None)

    for kw in (dict(prm="null"), dict(y=None), dict(state=None), dict(ws_ptr=None), dict(post=None), dict(out=None),
               dict(mean=fake), dict(mean2=fake)):
        assert call(**kw) == -1, kw
    for bad in (L.ImgShape(0, 3, 8, 8), L.ImgShape(1, 1, 8, 8), L.ImgShape(1, 3, 0, 8), L.ImgShape(1, 3, 8, 0),
                L.ImgShape(-1, 3, 8, 8)):
        assert call(shape=bad) == -1 and b"shape" in lib.psgla_last_error()
    inf, nan = float("inf"), float("nan")
    for field, values in (("ths", (0.0, -1.0, inf, nan)), ("tau", (0.0, -0.01, inf, nan)), ("rho", (0.0, 2.0, -1.0, nan)),
                          ("crit", (-1e-5, inf, nan)), ("n_it_max", (0, -5)), ("restart", (2, -1))):
        for v in values:
            prm = L.TVParams(0.1, 0.01, 1.99, 1e-5, 1000, 1)
            setattr(prm, field, v)
            assert call(prm=prm) == -1, (field, v)
            assert field.encode() in lib.psgla_last_error(), (field, lib.psgla_last_error())
    assert call(st=st - 1) == -4 and b"state" in lib.psgla_last_error()
    assert call(ws=ws - 1) == -4 and b"workspace" in lib.psgla_last_error()
