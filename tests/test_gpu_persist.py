"""
The persistent-CTA instantiations of the f = 1 tiled kernel (instances_g7.inc, DESIGN.md 4.1): one CTA per SM walks
the tiles, keeps the whole W search range in one box, reads the centre column from it and loads the next tile's box
during the epilogue.  The arithmetic per voxel is that of the one-tile-per-CTA kernel, so the two must agree bit for
bit -- and with the oracle.  NDNLM_PERSIST is read at plan creation.
"""
import numpy as np
import pytest

from helpers import sar_like, scaled_err

TOL32 = 1e-4
CFG3 = dict(r=(5, 5, 2), f=(1, 1, 1))


def _plan(shape, r, f, n_eff=-1):
    from nd_b200 import device
    return device.Plan(shape, r, f, 0.3, 0.6, n_eff)


def test_persistent_instantiation_is_chosen_for_cfg3_and_cfg2(monkeypatch):
    """One W pass with the trimmed exchange buffer fits the 227 KB a CTA may use; NDNLM_PERSIST=0 selects the
    two-pass kernel."""
    monkeypatch.delenv("NDNLM_PERSIST", raising=False)
    monkeypatch.delenv("NDNLM_DH", raising=False)
    for shape, r in (((4096, 4096, 32, 4), (5, 5, 2)), ((1024, 1024, 24, 4), (5, 5, 1))):
        p = _plan(shape, r, (1, 1, 1))
        assert p.kernel_name.endswith("(persist),ch=5,neff=false>[passes=1]"), p.kernel_name
        assert list(p.info.tile) == [14, 4, 30] and list(p.info.box)[0] == 26
        assert p.info.smem_bytes <= 232448
        assert "(persist)" in _plan(shape, r, (1, 1, 1), n_eff=20).kernel_name
    cfg3 = _plan((4096, 4096, 32, 4), (5, 5, 2), (1, 1, 1))
    assert cfg3.info.smem_bytes == 192256 + 38400 + 272          # box + 5 x 16 rows x 30 lanes x 16 B + mbarriers
    monkeypatch.setenv("NDNLM_PERSIST", "0")
    old = _plan((4096, 4096, 32, 4), (5, 5, 2), (1, 1, 1))
    assert "(persist)" not in old.kernel_name and old.kernel_name.endswith("[passes=2]"), old.kernel_name
    assert list(old.info.tile) == [14, 4, 30]
    monkeypatch.delenv("NDNLM_PERSIST")
    # other configurations keep their kernels: f = 2, float64, 2-D, V > 4, and boxes too large for one pass
    for shape, r, f, dt in (((256, 16384, 64, 4), (7, 7, 2), (2, 2, 2), np.float32),
                            ((210, 2048, 32, 4), (5, 5, 2), (1, 1, 1), np.float64),
                            ((1, 206, 500, 4), (0, 3, 3), (0, 1, 1), np.float32),
                            ((64, 256, 128, 6), (5, 5, 2), (1, 1, 1), np.float32),
                            ((64, 256, 128, 4), (8, 8, 2), (1, 1, 1), np.float32)):
        from nd_b200 import device
        p = device.Plan(shape, r, f, 0.3, 0.6, dtype=dt)
        assert p.is_tiled and "(persist)" not in p.kernel_name, p.kernel_name


def _both(dev_mod, monkeypatch, a, r, f, n_eff=-1):
    import torch
    outs, names = [], []
    for flag in ("0", "1"):
        monkeypatch.setenv("NDNLM_PERSIST", flag)
        plan = dev_mod.Plan(a.shape, r, f, 0.3, 0.6, n_eff)
        outs.append(plan.apply(torch.from_numpy(a).cuda()).cpu().numpy())
        names.append(plan.kernel_name)
    assert "(persist)" not in names[0], names
    return outs, names


@pytest.mark.gpu
@pytest.mark.parametrize("shape,persist", [
    ((30, 70, 16, 4), True),     # 3 x 4 x 3 = 36 tiles: fewer than SMs
    ((33, 61, 9, 4), True),      # no axis a tile multiple
    ((29, 32, 31, 4), True),
    ((29, 31, 32, 4), False),    # X = axis 2 (r_X = 2), R = axis 1 (r_R = 5): the one-pass box does not fit
    ((160, 210, 20, 4), True),   # 12 x 5 x 7 = 420 tiles: more than two per SM
])
def test_persistent_equals_one_tile_per_cta_bitwise(monkeypatch, c_oracle, shape, persist):
    from nd_b200 import device
    a = sar_like(shape, seed=41)
    (old, new), names = _both(device, monkeypatch, a, **CFG3)
    assert ("(persist)" in names[1]) == persist, names
    assert np.array_equal(old, new), (names, float(np.abs(old - new).max()))
    assert scaled_err(new, c_oracle.nlmeans(a, CFG3["r"], CFG3["f"], 0.3, 0.6, threads=8)) < TOL32


@pytest.mark.gpu
def test_persistent_neff_and_cfg2_radii_bitwise(monkeypatch, c_oracle):
    from nd_b200 import device
    a = sar_like((33, 61, 9, 4), seed=43)
    (old, new), names = _both(device, monkeypatch, a, n_eff=20.0, **CFG3)
    assert "(persist)" in names[1] and "neff=true" in names[1], names
    assert np.array_equal(old, new)
    assert scaled_err(new, c_oracle.nlmeans(a, CFG3["r"], CFG3["f"], 0.3, 0.6, 20.0, threads=8)) < TOL32
    b = sar_like((40, 64, 24, 3), seed=44)          # cfg2's radii, V = 3 (one zero lane in the variable group)
    (old, new), names = _both(device, monkeypatch, b, (5, 5, 1), (1, 1, 1))
    assert "(persist)" in names[1] and np.array_equal(old, new), names
    assert scaled_err(new, c_oracle.nlmeans(b, (5, 5, 1), (1, 1, 1), 0.3, 0.6, threads=8)) < TOL32


@pytest.mark.gpu
def test_persistent_sharded_and_plain_loader_bitwise(monkeypatch):
    """y shards (the shard / halo-exchange layer, two shards on one GPU) and the plain-load debugging loader give
    the unsharded TMA result bit for bit."""
    from nd_b200 import device
    from nd_b200._filters import _pixelwise_nlmeans_3d
    a = sar_like((80, 64, 12, 4), seed=45)
    monkeypatch.setenv("NDNLM_PERSIST", "1")
    assert "(persist)" in device.Plan(a.shape, CFG3["r"], CFG3["f"], 0.3, 0.6).kernel_name
    r, f = np.array(CFG3["r"], np.uint32), np.array(CFG3["f"], np.uint32)
    whole = np.full_like(a, np.nan)
    _pixelwise_nlmeans_3d(a, whole, r, f, 0.3, 0.6, pipeline=False)
    parts = np.full_like(a, np.nan)
    _pixelwise_nlmeans_3d(a, parts, r, f, 0.3, 0.6, shard_axis=0, devices=[0, 0], pipeline=False)
    assert np.array_equal(parts, whole)
    monkeypatch.setenv("NDNLM_LOADER", "ldg")
    ldg = np.full_like(a, np.nan)
    _pixelwise_nlmeans_3d(a, ldg, r, f, 0.3, 0.6, pipeline=False)
    assert np.array_equal(ldg, whole)
    monkeypatch.setenv("NDNLM_PERSIST", "0")
    monkeypatch.delenv("NDNLM_LOADER")
    old = np.full_like(a, np.nan)
    _pixelwise_nlmeans_3d(a, old, r, f, 0.3, 0.6, pipeline=False)
    assert np.array_equal(old, whole)
