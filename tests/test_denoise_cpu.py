"""The C restatement of the denoiser (tests/denoise_oracle.c), which tests/test_denoise.py holds the kernels to bit for bit:
its exp(-x), the fixed point of constant irradiance, the separation of surfaces with perpendicular normals and of hit and miss
pixels, and tiny frames.  CPU only."""
import numpy as np
import pytest

from denoise_ref import DenoiseOracle, synthetic_frame

EXP_REL_BOUND = 1e-5


@pytest.fixture(scope="module")
def oracle(rtnw, tmp_path_factory):
    return DenoiseOracle(rtnw, tmp_path_factory.mktemp("denoise_oracle"))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def test_exp_neg_is_within_its_bound(oracle):
    x = np.linspace(0, 88, 20_000_001, dtype=np.float32)[:-1]
    x = np.concatenate([x, np.float32(2.0) ** -np.arange(1, 140, dtype=np.float32)])  # tiny arguments down to denormals
    got = oracle.exp_neg(x).astype(np.float64)
    want = np.exp(-x.astype(np.float64))
    rel = np.abs(got - want) / want
    normal = want >= np.finfo(np.float32).tiny  # below it the result is a denormal, with up to one spacing (2^-149) more
    print(f"exp(-x): worst relative error {rel[normal].max():.3g} over [0, 88)")
    assert rel[normal].max() <= EXP_REL_BOUND, rel[normal].max()
    assert np.all(np.abs(got - want)[~normal] <= EXP_REL_BOUND * want[~normal] + 2.0 ** -149)
    assert oracle.exp_neg(np.float32([0.0]))[0] == 1.0
    edge = oracle.exp_neg(np.float32([88.0, 88.5, 1e30, np.inf, np.nan]))
    assert np.array_equal(bits(edge), bits(np.zeros(5, np.float32)))
    assert np.all(np.diff(oracle.exp_neg(np.linspace(0, 88, 100_001, dtype=np.float32))) <= 0)  # monotone on a coarse grid


@pytest.mark.parametrize("k", [0.5, 3.0])
def test_constant_irradiance_is_a_fixed_point(oracle, k):
    ns = 8
    color, aov = synthetic_frame(40, 30, ns, seed=1, zero_albedo_fraction=0)
    aov["albedo"] = np.maximum(aov["albedo"], np.float32(0.05 * ns))  # above the albedo floor everywhere
    color = (np.float32(k) * aov["albedo"]).astype(np.float32)
    out = oracle.denoise(color, aov, ns, iterations=5)
    want = color.astype(np.float64) / ns
    assert np.abs(out - want).max() <= 1e-6 * np.abs(want).max()
    assert np.all(np.abs(out - want) <= 1e-6 * want)


def _split_frame(nx, ny, ns):
    """all hits; normals (1,0,0) on the left half, (0,1,0) on the right"""
    color, aov = synthetic_frame(nx, ny, ns, seed=3, hit_fraction=1.0, zero_albedo_fraction=0)
    h = aov["hits"].astype(np.float32)
    n = np.zeros((ny, nx, 3), np.float32)
    n[:, : nx // 2, 0] = h[:, : nx // 2]
    n[:, nx // 2:, 1] = h[:, nx // 2:]
    aov["normal"] = n
    return color, aov


@pytest.mark.parametrize("iterations", [1, 5, 8])
def test_perpendicular_surfaces_do_not_mix(oracle, iterations):
    nx, ny, ns = 48, 20, 4
    color, aov = _split_frame(nx, ny, ns)
    a = oracle.denoise(color, aov, ns, iterations=iterations)
    other = color.copy()
    other[:, nx // 2:] *= np.float32(7.5)
    b = oracle.denoise(other, aov, ns, iterations=iterations)
    assert np.array_equal(bits(a[:, : nx // 2]), bits(b[:, : nx // 2]))
    assert not np.array_equal(bits(a[:, nx // 2:]), bits(b[:, nx // 2:]))


def test_hit_and_miss_pixels_do_not_mix(oracle):
    nx, ny, ns = 37, 29, 4
    color, aov = synthetic_frame(nx, ny, ns, seed=5, hit_fraction=0.6)
    miss = aov["hits"] == 0
    a = oracle.denoise(color, aov, ns)
    other = color.copy()
    other[~miss] *= np.float32(3.0)
    b = oracle.denoise(other, aov, ns)
    assert np.array_equal(bits(a[miss]), bits(b[miss]))
    # a black background: misses have no colour and no albedo, and stay exactly 0
    color[miss] = 0
    aov["albedo"][miss] = 0
    c = oracle.denoise(color, aov, ns)
    assert np.array_equal(bits(c[miss]), bits(np.zeros_like(c[miss])))
    assert np.all(np.isfinite(c)) and (c[~miss] > 0).any()


@pytest.mark.parametrize("nx, ny", [(1, 1), (1, 17), (17, 1), (2, 2)])
def test_tiny_frames(oracle, nx, ny):
    ns = 3
    color, aov = synthetic_frame(nx, ny, ns, seed=nx * 100 + ny, hit_fraction=0.5)
    out = oracle.denoise(color, aov, ns, iterations=8)
    assert out.shape == (ny, nx, 3) and np.all(np.isfinite(out))
    if nx * ny == 1:  # only the centre tap: the pixel's own mean
        assert np.allclose(out, color / ns, rtol=1e-6, atol=0)
