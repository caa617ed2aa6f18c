"""Chamfer op (SURVEY.md 8(f) rank 1): oracle self-consistency on the CPU, parity through the C-ABI on the GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import chamfer_oracle as CO


def _clouds(b, n, m, seed, dup=False):
    g = np.random.default_rng(seed)
    x1 = g.uniform(-1, 1, (b, n, 3)).astype(np.float32)
    x2 = g.uniform(-1, 1, (b, m, 3)).astype(np.float32)
    if dup and m > 8:          # exact duplicates in the target cloud: the smallest index has to win
        x2[:, m // 2:m // 2 + 4] = x2[:, 3:7]
        x1[:, :4] = x2[:, 3:7]
    return x1, x2


def test_oracle_matches_float64_cdist():
    x1, x2 = _clouds(2, 300, 411, 0, dup=True)
    d1, d2, i1, i2 = CO.chamfer_forward(x1, x2)
    for a, b, d, i in ((x1, x2, d1, i1), (x2, x1, d2, i2)):
        D = torch.cdist(torch.from_numpy(a).double(), torch.from_numpy(b).double()) ** 2
        dmin, _ = D.min(-1)
        assert np.allclose(d, dmin.numpy(), rtol=1e-5, atol=1e-9)
        picked = torch.gather(D, 2, torch.from_numpy(i.astype(np.int64))[..., None])[..., 0]
        assert np.allclose(picked.numpy(), dmin.numpy(), rtol=1e-5, atol=1e-9)
    assert (i1[:, :4] == np.arange(3, 7)).all()          # duplicates: first index wins (chamfer3D.cu:33,127)


def test_oracle_backward_matches_autograd():
    x1, x2 = _clouds(1, 64, 50, 1)
    d1, d2, i1, i2 = CO.chamfer_forward(x1, x2)
    g = np.random.default_rng(2)
    g1, g2 = g.normal(size=d1.shape).astype(np.float32), g.normal(size=d2.shape).astype(np.float32)
    gx1, gx2 = CO.chamfer_backward(x1, x2, g1, g2, i1, i2)
    t1 = torch.from_numpy(x1).double().requires_grad_(True)
    t2 = torch.from_numpy(x2).double().requires_grad_(True)
    D = torch.cdist(t1, t2) ** 2
    loss = (D.min(2)[0] * torch.from_numpy(g1).double()).sum() + (D.min(1)[0] * torch.from_numpy(g2).double()).sum()
    loss.backward()
    assert np.allclose(gx1, t1.grad.numpy(), rtol=1e-4, atol=1e-5)
    assert np.allclose(gx2, t2.grad.numpy(), rtol=1e-4, atol=1e-5)


def test_module_surface_and_argument_errors():
    from lidar4d_b200.chamfer import chamfer_3DDist, chamfer_3DFunction      # noqa: F401  (names of dist_chamfer_3D.py)
    f = chamfer_3DDist()
    with pytest.raises(ValueError):
        f(torch.zeros(1, 5, 2), torch.zeros(1, 5, 3))
    with pytest.raises(RuntimeError):
        f(torch.zeros(1, 5, 3), torch.zeros(1, 6, 3))       # CPU tensors: no fallback


CASES = [(1, 1024, 1024, 3, False), (2, 777, 1300, 4, True), (1, 1, 513, 5, False), (1, 700, 1, 6, False),
         (1, 20000, 15000, 7, True), (3, 50, 5000, 8, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("b,n,m,seed,dup", CASES)
def test_chamfer_forward_backward_gpu(b, n, m, seed, dup):
    from lidar4d_b200.chamfer import chamfer_3DDist
    dev = torch.device("cuda:0")
    x1, x2 = _clouds(b, n, m, seed, dup)
    rd1, rd2, ri1, ri2 = CO.chamfer_forward(x1, x2)
    t1 = torch.from_numpy(x1).to(dev).requires_grad_(True)
    t2 = torch.from_numpy(x2).to(dev).requires_grad_(True)
    d1, d2, i1, i2 = chamfer_3DDist()(t1, t2)
    assert i1.dtype == torch.int32 and d1.shape == (b, n) and d2.shape == (b, m)
    # distances: same fp32 expression as the reference kernel -> bit-exact against the fma-emulating oracle
    assert np.array_equal(d1.detach().cpu().numpy(), rd1) and np.array_equal(d2.detach().cpu().numpy(), rd2)
    assert np.array_equal(i1.cpu().numpy(), ri1) and np.array_equal(i2.cpu().numpy(), ri2)
    g = np.random.default_rng(seed + 100)
    g1, g2 = g.normal(size=rd1.shape).astype(np.float32), g.normal(size=rd2.shape).astype(np.float32)
    ((d1 * torch.from_numpy(g1).to(dev)).sum() + (d2 * torch.from_numpy(g2).to(dev)).sum()).backward()
    rg1, rg2 = CO.chamfer_backward(x1, x2, g1, g2, ri1, ri2)
    for got, ref in ((t1.grad, rg1), (t2.grad, rg2)):
        err = np.abs(got.cpu().numpy() - ref).max() / (np.abs(ref).max() + 1e-30)
        assert err < 1e-5, err


@pytest.mark.gpu
def test_chamfer_properties_full_size():
    """Size-independent properties at the flow-loss size (10^5 points): symmetry under swapping the clouds, zero
    distance and identity index for identical clouds, idempotence, gradient of sum(dist) sums to zero."""
    from lidar4d_b200.chamfer import chamfer_3DDist
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(0)
    a = (torch.rand(1, 100000, 3, generator=g) * 2 - 1).to(dev)
    bb = (torch.rand(1, 90000, 3, generator=g) * 2 - 1).to(dev)
    f = chamfer_3DDist()
    d1, d2, i1, i2 = f(a, bb)
    e2, e1, j2, j1 = f(bb, a)
    assert torch.equal(d1, e1) and torch.equal(d2, e2) and torch.equal(i1, j1) and torch.equal(i2, j2)
    s1, s2, k1, k2 = f(a, a.clone())
    assert float(s1.max()) == 0.0 and torch.equal(k1[0].long(), torch.arange(a.shape[1], device=dev))
    picked = ((a[0] - bb[0][i1[0].long()]) ** 2).sum(-1)
    assert torch.allclose(picked, d1[0], rtol=1e-5, atol=1e-9)
    a2 = a.clone().requires_grad_(True)
    b2 = bb.clone().requires_grad_(True)
    o1, o2, _, _ = f(a2, b2)
    (o1.sum() + o2.sum()).backward()
    tot = a2.grad.sum(1) + b2.grad.sum(1)
    assert float(tot.abs().max()) < 1e-2 * float(a2.grad.abs().sum())


# ---- the reference's OWN kernel (utils/chamfer3D/chamfer3D.cu compiled in place for sm_100a by oracle/build_ref.py) -------
def test_reference_extension_was_built():
    """oracle/_ref/chamfer_3D_ref.so is the reference's chamfer extension built by the committed recipe; it travels to
    the GPU box with the snapshot (the GPU box has no /root/reference)."""
    from oracle import build_ref
    if not os.path.exists(build_ref.REF) and not os.path.exists(build_ref.so_path()):
        pytest.skip("neither /root/reference nor a prebuilt oracle/_ref here")
    build_ref.build()                    # compiles in the build container when stale, no-op elsewhere
    assert os.path.exists(build_ref.so_path()), "run `python oracle/build_ref.py` in the build container"


REF_CASES = CASES + [(1, 4096, 4096, 11, True), (1, 60000, 50000, 12, False), (2, 1, 1, 13, False)]
REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "chamfer_ref.npz")


def chamfer_grad_inputs(b, n, m, seed):
    """Upstream gradients of dist1 / dist2 fed to both backward kernels."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, n, generator=g), torch.randn(b, m, generator=g)


def chamfer_grad_probes(size):
    """Fixed vector the stored gradients are projected on (no RNG: the same on every machine)."""
    return np.cos(np.arange(size, dtype=np.float64) * 0.618)


def _assert_bit_exact(fx, key, name, got):
    import hashlib
    a = np.ascontiguousarray(got).reshape(-1)
    pos = fx[f"{key}:pos:{name}"]
    assert np.array_equal(a[pos], fx[f"{key}:val:{name}"]), f"{name}: sampled entries differ from the reference kernel's"
    assert hashlib.sha256(a.tobytes()).hexdigest() == str(fx[f"{key}:sha:{name}"]), f"{name}: differs from the reference kernel's"


@pytest.mark.gpu
@pytest.mark.parametrize("b,n,m,seed,dup", REF_CASES)
def test_chamfer_bit_exact_against_reference_kernel(b, n, m, seed, dup):
    """Distances AND indices of l4d_chamfer_forward equal NmDistanceKernel's (chamfer3D.cu:11-133) bit for bit - also on
    exact duplicates (ties -> smallest index) - and the gradients equal NmDistanceGradKernel's (:154-174) to fp32
    atomics re-ordering.  This pins oracle/chamfer_oracle.py's assumed fma contraction as well.  The reference kernels'
    outputs on these inputs are stored in tests/golden/chamfer_ref.npz (make_golden.py --chamfer): distances and indices
    as a SHA-256 of the whole array, gradients as max |g|, a projection and a sample of points."""
    from lidar4d_b200.chamfer import chamfer_3DDist
    fx = np.load(REF_GOLDEN, allow_pickle=False)
    key = f"{b}x{n}x{m}_s{seed}"
    dev = torch.device("cuda:0")
    x1, x2 = _clouds(b, n, m, seed, dup)
    g1, g2 = chamfer_grad_inputs(b, n, m, seed)
    inputs = np.array([x1.sum(dtype=np.float64), x2.sum(dtype=np.float64), g1.double().sum().item(), g2.double().sum().item()])
    assert np.array_equal(inputs, fx[key + ":inputs"]), "the test inputs are not the ones the golden outputs were made from"
    t1 = torch.from_numpy(x1).to(dev).requires_grad_(True)
    t2 = torch.from_numpy(x2).to(dev).requires_grad_(True)
    d1, d2, i1, i2 = chamfer_3DDist()(t1, t2)
    for name, t in (("d1", d1), ("d2", d2), ("i1", i1), ("i2", i2)):
        _assert_bit_exact(fx, key, name, t.detach().cpu().numpy())
    o1, o2, oi1, oi2 = CO.chamfer_forward(x1, x2)                            # the numpy oracle agrees with the real kernel
    _assert_bit_exact(fx, key, "d1", o1)
    _assert_bit_exact(fx, key, "i2", oi2)
    ((d1 * g1.to(dev)).sum() + (d2 * g2.to(dev)).sum()).backward()
    for name, got in (("gx1", t1.grad), ("gx2", t2.grad)):
        a = got.cpu().numpy().reshape(-1, 3)
        tol = 1e-5 * float(fx[f"{key}:max:{name}"]) + 1e-12
        assert abs(float(np.abs(a).max()) - float(fx[f"{key}:max:{name}"])) <= tol, name
        assert float(np.abs(a[fx[f"{key}:pos:{name}"]] - fx[f"{key}:val:{name}"]).max()) <= tol, name
        probes = chamfer_grad_probes(a.size)
        assert abs(float(a.reshape(-1).astype(np.float64) @ probes) - float(fx[f"{key}:proj:{name}"])) <= tol * np.abs(probes).sum(), name
