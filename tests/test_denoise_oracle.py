"""CPU: the denoiser's oracle (oracle/denoise_api.cpp), which ptb_denoise is compared against, behaves as the spatial SVGF
filter should on synthetic sums: constant irradiance passes, the result stays inside its inputs' range, separated
regions exchange no energy, noise drops on piecewise-constant images, and the defaults are the documented values."""
import numpy as np
import pytest

from denoise_oracle import denoise


def make_sums(c, albedo, normal, depth, coverage, s_b=4, s_a=4):
    """Sums of s_b beauty samples of mean `c` and s_a AOV samples of the given means ((H, W, 8) AOV layout)."""
    h, w = c.shape[:2]
    aov = np.zeros((h, w, 8), np.float32)
    aov[..., 0:3] = albedo * s_a
    aov[..., 3] = coverage * s_a
    aov[..., 4:7] = normal * s_a
    aov[..., 7] = depth * coverage * s_a
    return (c * s_b).astype(np.float32), aov, s_b, s_a


def unit(v):
    v = np.asarray(v, np.float32)
    return v / np.linalg.norm(v)


def quadrants(h, w):
    """Four regions with their own normal (pairwise dot <= 0.8), depth, albedo and clean irradiance."""
    yy, xx = np.mgrid[0:h, 0:w]
    region = (yy >= h // 2).astype(int) * 2 + (xx >= w // 2).astype(int)
    normals = np.stack([unit((0, 0, 1)), unit((0.6, 0, 0.8)), unit((0, 0.6, 0.8)), unit((-0.6, 0, 0.8))])
    depth = np.float32([2.0, 3.0, 4.5, 6.0])[region]
    albedo = np.float32([[0.8, 0.5, 0.2], [0.3, 0.7, 0.9], [0.6, 0.6, 0.6], [0.9, 0.2, 0.4]])[region]
    irr = np.float32([0.5, 1.5, 3.0, 0.8])[region]
    return region, normals[region], depth, albedo, irr


def test_constant_irradiance_comes_out_unchanged():
    h, w = 40, 56
    region, n, z, a, _ = quadrants(h, w)
    c = (np.float32(0.7) * a).astype(np.float32)
    b, aov, sb, sa = make_sums(c, a, n, z, np.ones((h, w), np.float32))
    out = denoise(b, aov, sb, sa)
    assert np.all(np.isfinite(out))
    assert np.all(np.abs(out - c) <= 2e-6 * np.abs(c)), np.abs(out / c - 1).max()


def test_output_stays_within_the_input_range():
    rng = np.random.default_rng(3)
    h, w = 33, 47
    region, n, z, a, irr = quadrants(h, w)
    e = irr[..., None] * rng.uniform(0.2, 1.8, (h, w, 3)).astype(np.float32)
    b, aov, sb, sa = make_sums((e * a).astype(np.float32), a, n, z, np.ones((h, w), np.float32))
    d = np.maximum(aov[..., 0:3] / np.float32(sa), np.float32(1e-3))
    e_in = b * (np.float32(1) / np.float32(sb)) / d
    for it in (1, 3, 5):
        e_out = denoise(b, aov, sb, sa, iterations=it) / d
        for ch in range(3):
            lo, hi = e_in[..., ch].min(), e_in[..., ch].max()
            assert e_out[..., ch].min() >= lo * (1 - 1e-6) and e_out[..., ch].max() <= hi * (1 + 1e-6)


@pytest.mark.parametrize("split", ["normals", "hit_miss"])
def test_separated_regions_exchange_no_energy(split):
    """Left and right halves are told apart by orthogonal normals, or by hit against miss. One half holds a constant image,
    the other bright noise: the constant half comes out unchanged (the 3x3 variance prefilter reads across the edge, so
    its weights may change, but no tap of the other half enters its sums), and the bright half keeps its energy."""
    rng = np.random.default_rng(5)
    h, w = 24, 40
    half = w // 2
    for const_left in (True, False):
        n = np.zeros((h, w, 3), np.float32)
        cov = np.ones((h, w), np.float32)
        z = np.full((h, w), 3.0, np.float32)
        n[:, :half] = (0, 0, 1)
        if split == "normals":
            n[:, half:] = (1, 0, 0)
        else:  # the right half is a miss: no normal, no depth, no coverage
            cov[:, half:] = 0
            z[:, half:] = 0
        a = np.full((h, w, 3), 0.5, np.float32)
        c = rng.uniform(5.0, 50.0, (h, w, 3)).astype(np.float32)
        flat, noisy = (slice(0, half), slice(half, w)) if const_left else (slice(half, w), slice(0, half))
        c[:, flat] = 0.25
        out = denoise(*make_sums(c, a, n, z, cov))
        assert np.all(np.abs(out[:, flat] - np.float32(0.25)) <= 2e-6 * 0.25), np.abs(out[:, flat] - 0.25).max()
        assert out[:, noisy].min() >= c[:, noisy].min() * (1 - 1e-6)


@pytest.mark.parametrize("seed", [1, 2])
def test_noise_drops_on_piecewise_constant_images(seed):
    rng = np.random.default_rng(seed)
    h, w = 64, 96
    region, n, z, a, irr = quadrants(h, w)
    clean = (irr[..., None] * a).astype(np.float32)
    noisy = (clean * (1 + 0.3 * rng.standard_normal((h, w, 3)))).astype(np.float32)
    b, aov, sb, sa = make_sums(noisy, a, n, z, np.ones((h, w), np.float32))
    out = denoise(b, aov, sb, sa)
    err_noisy = np.sqrt(np.mean((noisy - clean) ** 2))
    err_out = np.sqrt(np.mean((out - clean) ** 2))
    assert err_out * 10 <= err_noisy, (err_noisy, err_out)  # about 25x on both seeds


def test_defaults_equal_their_explicit_values():
    rng = np.random.default_rng(9)
    h, w = 30, 50
    region, n, z, a, irr = quadrants(h, w)
    noisy = (irr[..., None] * a * (1 + 0.5 * rng.standard_normal((h, w, 3)))).astype(np.float32)
    b, aov, sb, sa = make_sums(noisy, a, n, z, np.ones((h, w), np.float32))
    d = denoise(b, aov, sb, sa)
    e = denoise(b, aov, sb, sa, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0)
    assert np.array_equal(d.view(np.uint32), e.view(np.uint32))
    assert not np.array_equal(d, denoise(b, aov, sb, sa, iterations=2))
