"""CPU tests of the drop-in boundary: the C-ABI library builds for sm_100a, loads without a GPU and exports
every symbol include/egs_raster.h declares; argument validation fails loudly; nothing routes to the oracle."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def _declared_symbols():
    text = (ROOT / "include" / "egs_raster.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(egs_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from easy_gaussian_splatting_b200 import _lib
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/egs_raster.h but not exported"
    assert set(_lib.EXPORTED_SYMBOLS) == set(declared), "Python binding table and header disagree"
    assert lib.egs_abi_version() == 1


def test_workspace_queries_and_argument_errors_without_gpu():
    from easy_gaussian_splatting_b200 import _lib
    lib = _lib.load()
    assert lib.egs_exclusive_scan_workspace_bytes(1_000_000) >= 8 * (1_000_000 // 2048)
    b6 = lib.egs_radix_sort_workspace_bytes(10_000_000, 45)
    b8 = lib.egs_radix_sort_workspace_bytes(10_000_000, 64)
    assert 0 < b6 < b8
    # invalid arguments are rejected before any launch (works without a device)
    rc = lib.egs_radix_sort_pairs_u64_u32(-1, None, None, None, None, 45, None, 0, None, None)
    assert rc == -1 and b"n=-1" in lib.egs_last_error_string()
    rc = lib.egs_rasterize_fwd(1, 0, 0, None, None, None, None, 100, 100, 3, 3, None, None, None, None, None)
    assert rc == -1 and b"tile grid" in lib.egs_last_error_string()
    rc = lib.egs_projection_fwd(1, 10, None, None, None, None, None, 16, 5, 0, None, None, 64, 64, 0.3, 0.01, 1e10, 0.0,
                                16, 4, 4, None, None, None, None, None, None, None, None, None)
    assert rc == -1 and b"sh_degree" in lib.egs_last_error_string()


def test_projection_backward_rejects_too_few_sh_coefficients_without_gpu():
    """K < (sh_degree + 1)^2 would make the backward kernels read past each SH row: every backward entry rejects it
    before any launch, as the forward does."""
    from easy_gaussian_splatting_b200 import _lib
    lib = _lib.load()
    n0 = lib.egs_kernel_launch_count()
    fake = ctypes.c_void_p(0x1000)  # a non-null v_viewmats that is never touched
    for K, deg in ((9, 3), (4, 2), (1, 1), (15, 3)):
        rc = lib.egs_projection_bwd(1, 10, None, None, None, None, K, deg, 0, None, None, 64, 64, 0.3, None, None, None,
                                    None, None, None, None, None, None, None, None)
        assert rc == -1 and f"K={K} too small".encode() in lib.egs_last_error_string(), (K, deg)
        rc = lib.egs_projection_bwd_antialiased(1, 10, None, None, None, None, None, K, deg, 0, None, None, 64, 64, 0.3,
                                                None, None, None, None, None, None, None, None, None, None, None)
        assert rc == -1 and f"K={K} too small".encode() in lib.egs_last_error_string(), (K, deg)
        rc = lib.egs_projection_bwd_viewmats(1, 10, None, None, None, None, None, K, deg, 0, None, None, 64, 64, 0.3,
                                             None, None, None, None, None, None, None, None, None, None, 0, fake, None, 0,
                                             None)
        assert rc == -1 and f"K={K} too small".encode() in lib.egs_last_error_string(), (K, deg)
    assert lib.egs_kernel_launch_count() == n0


def test_product_never_imports_the_oracle_and_has_no_cpu_path():
    pkg = ROOT / "easy_gaussian_splatting_b200"
    for f in pkg.rglob("*.py"):
        src = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+[^\n]*\boracle\b", src, flags=re.M), f"{f} imports the oracle"
        assert "gsplat_oracle" not in src, f"{f} references the oracle module"
    from easy_gaussian_splatting_b200 import rasterization
    from easy_gaussian_splatting_b200.synthetic import make_scene
    sc = make_scene("blob", 10, 16, 16, 10.0, 0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rasterization(sc.means, sc.quats, sc.scales, sc.opacities, sc.colors, sc.viewmats, sc.Ks, 16, 16, sh_degree=3, packed=False)


def test_signature_matches_gsplat_1_0_0():
    import inspect
    from easy_gaussian_splatting_b200 import rasterization
    params = list(inspect.signature(rasterization).parameters.items())
    names = [n for n, _ in params]
    assert names == ["means", "quats", "scales", "opacities", "colors", "viewmats", "Ks", "width", "height", "near_plane",
                     "far_plane", "radius_clip", "eps2d", "sh_degree", "packed", "tile_size", "backgrounds", "render_mode",
                     "sparse_grad", "absgrad", "rasterize_mode", "channel_chunk"]
    d = {n: p.default for n, p in params}
    assert (d["near_plane"], d["far_plane"], d["radius_clip"], d["eps2d"]) == (0.01, 1e10, 0.0, 0.3)
    assert d["sh_degree"] is None and d["packed"] is True and d["tile_size"] == 16 and d["backgrounds"] is None
    assert d["render_mode"] == "RGB" and d["absgrad"] is False and d["rasterize_mode"] == "classic"


def test_input_validation_messages():
    from easy_gaussian_splatting_b200.rendering import _check_inputs
    N, C = 5, 1
    f = lambda *s: torch.zeros(*s)
    good = dict(means=f(N, 3), quats=f(N, 4), scales=f(N, 3), opacities=f(N), colors=f(N, 16, 3), viewmats=f(C, 4, 4),
                Ks=f(C, 3, 3), sh_degree=3, backgrounds=None)
    for key, bad in (("means", f(N, 2)), ("quats", f(N, 3)), ("opacities", f(N, 1)), ("viewmats", f(C, 3, 4)), ("colors", f(N, 4, 3))):
        kw = dict(good)
        kw[key] = bad
        with pytest.raises((ValueError, NotImplementedError)):
            _check_inputs(**kw)
