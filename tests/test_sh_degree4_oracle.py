"""CPU tests of the degree-4 SH reference (tests/sh_degree4_reference.py): its 25 basis functions are the real
spherical harmonics of the lower degrees' convention, built independently from scipy's complex Y_l^m, and they are
orthonormal on the sphere."""
import numpy as np
import pytest
import torch
from scipy.special import sph_harm_y

from oracle import gsplat_oracle as O
from tests.sh_degree4_reference import sh_basis4


def _random_dirs(n, seed):
    d = torch.randn(n, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    return d * torch.rand(n, 1, generator=torch.Generator().manual_seed(seed + 1), dtype=torch.float64).add(0.1) * 3


def _complex_construction(degree, dirs):
    """Real SH from scipy's complex Y_l^m (Condon-Shortley phase included): sqrt(2) Re Y_l^m for m > 0,
    sqrt(2) Im Y_l^|m| for m < 0, Y_l^0 for m = 0, each band ordered m = -l..l."""
    d = dirs.numpy()
    d = d / np.linalg.norm(d, axis=-1, keepdims=True)
    theta = np.arccos(np.clip(d[:, 2], -1.0, 1.0))
    phi = np.arctan2(d[:, 1], d[:, 0])
    out = []
    for l in range(degree + 1):
        for m in range(-l, l + 1):
            y = sph_harm_y(l, abs(m), theta, phi)
            out.append(np.sqrt(2.0) * y.real if m > 0 else np.sqrt(2.0) * y.imag if m < 0 else y.real)
    return torch.from_numpy(np.stack(out, -1))


def test_construction_reproduces_the_oracle_degrees_0_to_3():
    dirs = _random_dirs(2000, 0)
    assert torch.allclose(_complex_construction(3, dirs), O.sh_basis(3, dirs), rtol=0, atol=1e-12)


@pytest.mark.parametrize("seed", [1, 2])
def test_degree4_basis_matches_the_complex_construction(seed):
    dirs = _random_dirs(2000, seed)
    got, ref = sh_basis4(dirs), _complex_construction(4, dirs)
    assert got.shape == (2000, 25)
    err = (got - ref).abs().amax(0)
    assert torch.all(err <= 1e-12), err
    assert torch.equal(got[:, :16], O.sh_basis(3, dirs))  # bands 0..3 are the oracle's, bit for bit


def test_degree4_basis_is_orthonormal():
    """Gauss-Legendre in cos(theta) (10 nodes) x 20 uniform phi: exact for the degree-8 products of two functions."""
    t, w = np.polynomial.legendre.leggauss(10)
    phi = np.arange(20) * (2 * np.pi / 20)
    ct, ph = np.meshgrid(t, phi, indexing="ij")
    st = np.sqrt(1.0 - ct ** 2)
    dirs = torch.from_numpy(np.stack([st * np.cos(ph), st * np.sin(ph), ct], -1).reshape(-1, 3))
    wt = torch.from_numpy(np.repeat(w, 20) * (2 * np.pi / 20))
    Y = sh_basis4(dirs)
    gram = (Y * wt[:, None]).T @ Y
    assert torch.allclose(gram, torch.eye(25, dtype=torch.float64), rtol=0, atol=1e-12), (gram - torch.eye(25)).abs().max()


def test_degree4_basis_is_scale_invariant():
    dirs = _random_dirs(100, 5)
    assert torch.allclose(sh_basis4(dirs), sh_basis4(dirs * 7.5), rtol=0, atol=1e-13)
