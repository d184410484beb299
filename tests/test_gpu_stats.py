"""GPU parity tests for kernel 3 (GAE + advantage normalisation, Welford) and kernel 4 (row gather), through the
C-ABI, against the CPU oracle.  GAE is fp32 arithmetic in torch's operation order: unnormalised advantages and value
targets must match the oracle bit for bit; the normalised advantages (whole-tensor mean / unbiased std) within
1e-5 relative, the tolerance north_star states for GAE and normalisation statistics."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _gae_gpu(r, v, active, gamma, lamda, norm, time_major):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    if time_major:
        T, B, N = r.shape
    else:
        B, T, N = r.shape
    adv = torch.empty_like(r)
    vt = torch.empty_like(r)
    ws = torch.zeros(int(L.marl_gae_workspace_bytes(B, T, N)), dtype=torch.uint8, device=r.device)
    _lib.check(L.marl_gae(B, T, N, _lib.ptr(r), _lib.ptr(v), _lib.ptr(active), 1 if time_major else 0,
                          ctypes.c_float(gamma), ctypes.c_float(gamma * lamda), 1 if norm else 0, _lib.ptr(adv),
                          _lib.ptr(vt), _lib.ptr(ws), _lib.stream_ptr()), "marl_gae")
    torch.cuda.synchronize()
    return adv, vt


@pytest.mark.parametrize("B,T,N", [(3, 7, 4), (64, 150, 8), (257, 33, 15)])
def test_gae_matches_oracle(oracle, B, T, N):
    rng = np.random.default_rng(B * 1000 + T)
    r = rng.normal(0, 1, (B, T, N)).astype(np.float32)
    v = rng.normal(0, 1, (B, T + 1, N)).astype(np.float32)
    active = (rng.random((B, T, N)) < 0.9).astype(np.float32)
    adv0, vt0 = oracle.gae(r, v, active, 0.99, 0.95, use_adv_norm=False)
    adv1, _ = oracle.gae(r, v, active, 0.99, 0.95, use_adv_norm=True)
    rd, vd, ad = (torch.from_numpy(x).cuda() for x in (r, v, active))
    # reference layout [B,T,N]
    adv, vt = _gae_gpu(rd, vd, ad, 0.99, 0.95, False, False)
    assert np.array_equal(adv.cpu().numpy(), adv0) and np.array_equal(vt.cpu().numpy(), vt0)
    advn, vtn = _gae_gpu(rd, vd, ad, 0.99, 0.95, True, False)
    assert np.array_equal(vtn.cpu().numpy(), vt0)
    np.testing.assert_allclose(advn.cpu().numpy(), adv1, rtol=1e-5, atol=1e-6)
    # time-major arena layout [T,B,N]: same numbers, permuted
    rt, vtm, at = (x.transpose(0, 1).contiguous() for x in (rd, vd, ad))
    adv_t, vt_t = _gae_gpu(rt, vtm, at, 0.99, 0.95, True, True)
    assert torch.equal(adv_t.transpose(0, 1), advn) and torch.equal(vt_t.transpose(0, 1), vtn)


def test_gae_properties_at_full_size():
    """config-2 size (4096 x 150 x 8): linear in r when v=0 and no normalisation; normalised output has zero mean and
    unit (unbiased) std; inactive samples are exactly zero."""
    B, T, N = 4096, 150, 8
    g = torch.Generator(device="cuda").manual_seed(0)
    r = torch.randn(T, B, N, device="cuda", generator=g)
    v = torch.zeros(T + 1, B, N, device="cuda")
    active = torch.ones(T, B, N, device="cuda")
    a1, _ = _gae_gpu(r, v, active, 0.99, 0.95, False, True)
    a2, _ = _gae_gpu(2 * r, v, active, 0.99, 0.95, False, True)
    assert torch.equal(a2, 2 * a1)                       # exact: scaling by 2 commutes with every rounding
    active[:, ::7] = 0
    an, _ = _gae_gpu(r, v, active, 0.99, 0.95, True, True)
    assert (an[:, ::7] == 0).all()
    raw, _ = _gae_gpu(r, v, active, 0.99, 0.95, False, True)
    ref = (raw - raw.mean()) / (raw.std() + 1e-5) * active
    torch.testing.assert_close(an, ref, rtol=1e-5, atol=1e-6)


def test_welford_kernel_matches_oracle(oracle):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    B, N, steps = 129, 15, 12
    rng = np.random.default_rng(1)
    n = torch.zeros(B, dtype=torch.int64, device="cuda")
    mean = torch.zeros(B, N, dtype=torch.float64, device="cuda")
    S = torch.zeros_like(mean)
    sd = torch.zeros_like(mean)
    out = torch.zeros(B, N, dtype=torch.float32, device="cuda")
    wfs = [oracle.Welford(N) for _ in range(B)]
    for t in range(steps):
        x = rng.integers(-3, 2, (B, N)).astype(np.int32)
        xd = torch.from_numpy(x).cuda()
        _lib.check(L.marl_welford_update(B, N, _lib.ptr(xd), _lib.ptr(n), _lib.ptr(mean), _lib.ptr(S), _lib.ptr(sd),
                                         _lib.ptr(out), 1, _lib.stream_ptr()))
        exp = np.stack([wfs[b](x[b]) for b in range(B)])
        assert np.array_equal(out.cpu().numpy(), exp), t
    # update=False leaves the statistics alone
    before = mean.clone()
    _lib.check(L.marl_welford_update(B, N, _lib.ptr(xd), _lib.ptr(n), _lib.ptr(mean), _lib.ptr(S), _lib.ptr(sd),
                                     _lib.ptr(out), 0, _lib.stream_ptr()))
    assert torch.equal(mean, before) and int(n[0]) == steps


@pytest.mark.parametrize("row_elems,dtype", [(8 * 4, torch.float32), (150 * 8 * 176, torch.float32), (7, torch.int32), (150 * 8 * 6, torch.int32),
                                             (33, torch.uint8), (3 * 33, torch.uint8)])
def test_gather_rows(row_elems, dtype):
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    Bsrc, n = 97, 41
    g = torch.Generator(device="cuda").manual_seed(3)
    src = torch.randint(-1000, 1000, (Bsrc, row_elems), device="cuda", generator=g).to(dtype)
    idx = torch.randint(0, Bsrc, (n,), device="cuda", generator=g)
    dst = torch.empty(n, row_elems, dtype=dtype, device="cuda")
    _lib.check(L.marl_gather_rows(_lib.ptr(src), _lib.ptr(dst), _lib.ptr(idx), n, row_elems * src.element_size(), Bsrc,
                                  _lib.stream_ptr()))
    assert torch.equal(dst, src[idx])
    # sequential index lists (the reference's SequentialSampler) are the identity on a slice
    seq = torch.arange(10, 30, device="cuda")
    dst2 = torch.empty(20, row_elems, dtype=dtype, device="cuda")
    _lib.check(L.marl_gather_rows(_lib.ptr(src), _lib.ptr(dst2), _lib.ptr(seq), 20, row_elems * src.element_size(), Bsrc,
                                  _lib.stream_ptr()))
    assert torch.equal(dst2, src[10:30])


def test_reward_scaling_matches_reference():
    """RewardScaling (DHGN/normalization.py:38-52) on the f64 Welford entry against the reference's own outputs
    (tests/golden/reward_scaling.npz, oracle/gen_golden_reward_scaling.py): two episodes with a reset() between them."""
    from conftest import golden
    from distributed_multi_agent_reinforcement_learning_b200.normalization import RewardScaling
    fx = golden("reward_scaling")
    x, T = fx["x"], fx["x"].shape[0] // 2
    rs = RewardScaling(shape=x.shape[1], gamma=float(fx["gamma"]))
    for t in range(2 * T):
        if t == T:
            rs.reset()
        np.testing.assert_allclose(rs(x[t]), fx["out"][t], rtol=1e-12, atol=0)
    ms = rs.running_ms
    assert ms.n == int(fx["n"])
    np.testing.assert_allclose(ms.mean, fx["mean"], rtol=1e-12)
    np.testing.assert_allclose(ms.S, fx["S"], rtol=1e-12)
    np.testing.assert_allclose(ms.std, fx["std"], rtol=1e-12)
    np.testing.assert_allclose(rs.R, fx["R"], rtol=1e-14)
