"""SURVEY.md §8(f) N3: TrowbridgeReitz material, Checkered / Perlin / Image textures, image decoding — oracle side (CPU).

reference test                                                       -> here
  bxdfs/trowbridge_reitz_vndf.rs:156-184 chi^2 isotropic_h / isotropic / isotropic_non_local -> test_tr_vndf_chi_squared
  bxdfs/trowbridge_reitz.rs:128-143 g1_cos_test                      -> test_tr_integrals[g1_cos]
  bxdfs/trowbridge_reitz.rs:145-163 projected_area (local, non-local)-> test_tr_integrals[projected_area*]
  bxdfs/trowbridge_reitz.rs:165-186 weak_furnace_test                -> test_tr_integrals[weak_furnace]
  bxdfs/trowbridge_reitz.rs:188-230 g2_test (local, non-local)       -> test_tr_integrals[g2*]
The reference draws alpha / incoming at random per run; here they are fixed grids of the same ranges.
Perlin / Image / Checkered have no reference tests ("parity unpinned" there): checked against independent numpy
restatements of textures/mod.rs.
"""
import os
import struct
import zlib

import numpy as np
import pytest

from test_oracle_kats import _chi2_sphere


def _wi(cos_theta, phi):
    """-generate_wi(): a unit vector in the upper hemisphere (spherical_sampling.rs:237-242)."""
    s = np.sqrt(1 - cos_theta * cos_theta)
    return np.array([s * np.cos(phi), s * np.sin(phi), cos_theta], np.float32)


def _to_world(z, v):
    """Coordinate::new_from_z(z).to_coord(v) (utility/coord.rs:10-30)."""
    z = z.astype(np.float64)
    x = np.array([-z[2], 0, z[0]]) / np.hypot(z[0], z[2]) if abs(z[0]) > abs(z[1]) else np.array([0, z[2], -z[1]]) / np.hypot(z[1], z[2])
    y = np.cross(x, z)
    return (v[0] * x + v[1] * y + v[2] * z).astype(np.float32)


def _sphere_grid(n_theta=480, n_phi=960):
    """midpoint quadrature nodes + solid-angle weights over the sphere (integrate_over_sphere, spherical_sampling.rs:39-62)"""
    th = (np.arange(n_theta) + 0.5) * np.pi / n_theta
    ph = (np.arange(n_phi) + 0.5) * 2 * np.pi / n_phi
    T, P = np.meshgrid(th, ph, indexing="ij")
    d = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], -1).reshape(-1, 3).astype(np.float32)
    w = (np.sin(T) * (np.pi / n_theta) * (2 * np.pi / n_phi)).reshape(-1)
    return d, w


@pytest.mark.parametrize("which", ["h", "local", "world"])
@pytest.mark.parametrize("alpha,cos_i", [(0.15, 0.9), (0.5, 0.6), (0.9, 0.25)])
def test_tr_vndf_chi_squared(orc, which, alpha, cos_i):
    incoming = _wi(cos_i, 1.1)
    normal = np.array([0, 0, 1], np.float32)
    mode = {"h": orc.TR_H, "local": orc.TR_LOCAL, "world": orc.TR_WORLD}[which]
    if which == "world":
        normal = orc.random_unit_vectors(1, seed=17)[0]
        incoming = _to_world(normal, incoming)            # to_local.to_coord(-generate_wi())
    dirs = orc.tr_sample(alpha, incoming, 300_000, seed=5, which=mode, normal=normal)
    assert np.allclose(np.linalg.norm(dirs, axis=1), 1, atol=1e-4)
    p, mass_err = _chi2_sphere(dirs, lambda d: orc.tr_pdf(alpha, incoming, d, which=mode, normal=normal), n_theta=40, n_phi=80)
    assert mass_err < 5e-3      # the pdf integrates to 1 (test_spherical_pdf panics beyond 0.001 with its finer quadrature)
    assert p > 0.01 / 10


@pytest.mark.parametrize("alpha", [0.2, 0.5, 0.95])
@pytest.mark.parametrize("cos_a", [0.95, 0.5, 0.15])
def test_tr_integrals(orc, alpha, cos_a):
    d, w = _sphere_grid()
    a = _wi(cos_a, 0.7)
    z = np.array([0, 0, 1], np.float32)
    # g1_cos_test: integral of G1 * max(a.h, 0) * D(h) = cos(theta_a)
    assert abs(np.sum(orc.tr_integrand(alpha, a, d, 0) * w) - cos_a) < 2e-3
    # projected_area_test_local / non_local: integral of D(h) (h.n) = 1
    assert abs(np.sum(orc.tr_integrand(alpha, a, d, 1) * w) - 1.0) < 2e-3
    n = orc.random_unit_vectors(1, seed=3)[0]
    assert abs(np.sum(orc.tr_integrand(alpha, a, d, 1, normal=n) * w) - 1.0) < 2e-3
    # weak_furnace_test: integral of G1 D / (4 |wo.n|) = 1
    assert abs(np.sum(orc.tr_integrand(alpha, a, d, 2) * w) - 1.0) < 3e-3
    # g2_test: integral of G2 D / (4 |a.n|) <= 1
    assert np.sum(orc.tr_integrand(alpha, a, d, 3) * w) <= 1.0 + 1e-3
    assert np.all(np.isfinite(orc.tr_integrand(alpha, a, d, 3, normal=z)))


def _tr_scene(ptb, alpha=0.3, ior=(1.5, 1.5, 1.5), metallic=0.0):
    s = ptb.HostScene()
    t = s.add_texture(ptb.TEX_SOLID, (0.9, 0.6, 0.3))
    m = s.add_material(ptb.MAT_TROWBRIDGE_REITZ, t, alpha, ior=ior, metallic=metallic)
    s.add_sphere((0, 0, 0), 1.0, m)
    s.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 40)
    s.set_sky(t, (0, 0))
    return s, m


def test_tr_material_methods(ptb, orc):
    """materials/trowbridge_reitz.rs:38-88: eval == eval_over_pdf * pdf away from the zero set; fresnel lerps to the
    texture colour with `metallic`; pdf 0 -> INFINITY."""
    for metallic in (0.0, 0.7, 1.0):
        hs, m = _tr_scene(ptb, 0.3, (1.5, 1.5, 1.5), metallic)
        o = orc.OracleScene(hs)
        n = np.array([0, 0, 1], np.float32)
        rng = np.random.default_rng(1)
        for _ in range(50):
            wo_out = _wi(rng.uniform(0.2, 1), rng.uniform(0, 6.28))       # pointing away from the surface
            wi = _wi(rng.uniform(0.2, 1), rng.uniform(0, 6.28))
            pdf, ev, eop = o.material_terms(m, n, (0, 0, 1), -wo_out, wi)  # the integrator's wo points INTO the surface
            assert pdf > 0 and np.all(np.isfinite(ev)) and np.all(ev >= 0)
            # eval / pdf == f g2 d / (4 |wo.n| wi.n) * 4 wo.h / (g1 max(wo.h,0) d / wo.n) == f g2 / g1 / wi.n ... the
            # reference's eval carries the 1/(wi.n) of the BRDF while eval_over_scattering_pdf does not carry cos(wi)
            assert np.allclose(ev / pdf, eop / wi[2], rtol=2e-3, atol=1e-6)
        # below the horizon: eval is zero and the pdf of an impossible direction is reported as infinity
        pdf, ev, eop = o.material_terms(m, n, (0, 0, 1), -_wi(0.5, 0.3), -_wi(0.5, 2.0))
        assert np.all(ev == 0) and np.all(eop == 0)
    hs, m = _tr_scene(ptb, 0.3, (1.5, 1.5, 1.5), 1.0)
    o = orc.OracleScene(hs)
    # normal incidence, metallic = 1: F = F0 = texture colour
    _, _, eop = o.material_terms(m, (0, 0, 1), (0, 0, 1), (0, 0, -1), (0, 0, 1))
    assert np.allclose(eop, (0.9, 0.6, 0.3), atol=1e-5)


# ---------------------------------------------------------------------------------------------- textures
def test_checkered_and_lerp(ptb, orc):
    s = ptb.HostScene()
    tc = s.add_texture(ptb.TEX_CHECKERED, (1, 0, 0), (0, 0, 1))
    m = s.add_material(ptb.MAT_LAMBERTIAN, tc, 0.5)
    s.add_sphere((0, 0, 0), 1, m)
    s.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 40)
    s.set_sky(tc, (0, 0))
    o = orc.OracleScene(s)
    rng = np.random.default_rng(0)
    for p in rng.uniform(-2, 2, (200, 3)).astype(np.float32):
        sign = np.sin(np.float32(10) * p[0]) * np.sin(np.float32(10) * p[1]) * np.sin(np.float32(10) * p[2])
        if abs(sign) < 1e-4:
            continue
        assert np.array_equal(o.texture_colour(tc, (0, 0, 1), p), (1, 0, 0) if sign > 0 else (0, 0, 1))


def _perlin_numpy(words, p):
    ran = words[:256]
    perm = words[256:].view(np.uint32).reshape(3, 256)
    f = np.floor(p)
    u, v, w = (p - f).astype(np.float32)
    i, j, k = f.astype(np.int64)
    uu, vv, ww = (t * t * (3 - 2 * t) for t in (u, v, w))
    val = np.float32(0)
    for idx in range(8):
        di, dj, dk = idx // 4, (idx // 2) % 2, idx % 2
        r = ran[perm[0][(i + di) & 255] ^ perm[1][(j + dj) & 255] ^ perm[2][(k + dk) & 255]]
        val += (di * uu + (1 - di) * (1 - uu)) * (dj * vv + (1 - dj) * (1 - vv)) * (dk * ww + (1 - dk) * (1 - ww)) * \
            (r * (u - di) + r * (v - dj) + r * (w - dk))
    return 0.5 * (1 + val)


def test_perlin(ptb, orc):
    s = ptb.HostScene()
    tp = s.add_perlin_texture(seed=7)
    _, _, words = s.texture_data[tp]
    perm = words[256:].view(np.uint32).reshape(3, 256)
    for k in range(3):
        assert sorted(perm[k]) == list(range(256))          # generate_perm: a permutation of 0..255
    assert not np.array_equal(perm[0], perm[1])
    assert np.all(np.abs(words[:256]) <= 1.0)                # gen_range(-1.0..1.0)
    assert abs(float(words[:256].mean())) < 0.15
    s2 = ptb.HostScene()
    assert np.array_equal(s2.texture_data[s2.add_perlin_texture(seed=7)][2], words)   # pure function of the seed
    m = s.add_material(ptb.MAT_LAMBERTIAN, tp, 0.5)
    s.add_sphere((0, 0, 0), 1, m)
    s.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 40)
    s.set_sky(tp, (0, 0))
    o = orc.OracleScene(s)
    rng = np.random.default_rng(2)
    for p in rng.uniform(-300, 300, (300, 3)).astype(np.float32):
        c = o.texture_colour(tp, (0, 0, 1), p)
        assert c[0] == c[1] == c[2]
        assert abs(c[0] - _perlin_numpy(words, p)) < 1e-5


def test_image_texture_lookup(ptb, orc):
    rng = np.random.default_rng(3)
    img = rng.uniform(0, 1, (7, 13, 3)).astype(np.float32)
    s = ptb.HostScene()
    ti = s.add_image_texture(img)
    m = s.add_material(ptb.MAT_LAMBERTIAN, ti, 0.5)
    s.add_sphere((0, 0, 0), 1, m)
    s.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 40)
    s.set_sky(ti, (8, 4))
    o = orc.OracleScene(s)
    for d in orc.random_unit_vectors(500, seed=4):
        phi = np.arctan2(d[1], d[0]) + np.pi
        theta = np.arccos(d[2])
        fx, fy = 12 * (phi / (2 * np.pi)), 6 * (theta / np.pi)
        if min(abs(fx - round(fx)), abs(fy - round(fy))) < 1e-3:
            continue  # a texel boundary: f32 vs f64 may round either way
        x, y = int(fx), int(fy)                                            # dim = (w-1, h-1): textures/mod.rs:232
        assert np.array_equal(o.texture_colour(ti, d), img[y, x])
    # the sky distribution is built from the image (sky.rs:20-37): brighter rows/columns get more pdf mass
    ycdf, xcdf, ypdf, xpdf = o.sky_table()
    assert abs(ypdf.sum() - 1) < 1e-5 and np.allclose(xpdf.reshape(4, 8).sum(axis=1), 1, atol=1e-5)


def _png_bytes(arr, bit_depth=8, colour_type=2, level=6):
    """arr: (H, W, C) uint8/uint16. Real (compressed, filtered) PNG for the decoder test."""
    h, w, c = arr.shape
    raw = bytearray()
    prev = np.zeros((w * c * (bit_depth // 8),), np.uint8)
    for y in range(h):
        row = (arr[y].astype(">u2").tobytes() if bit_depth == 16 else arr[y].astype(np.uint8).tobytes())
        row = np.frombuffer(row, np.uint8)
        ft = y % 3  # None, Sub, Up
        bpp = c * (bit_depth // 8)
        if ft == 0:
            out = row
        elif ft == 1:
            shifted = np.concatenate([np.zeros(bpp, np.uint8), row[:-bpp]])
            out = (row.astype(np.int16) - shifted).astype(np.uint8)
        else:
            out = (row.astype(np.int16) - prev).astype(np.uint8)
        raw.append(ft)
        raw += out.tobytes()
        prev = row

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xFFFFFFFF)
    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, bit_depth, colour_type, 0, 0, 0))
            + chunk(b"IDAT", zlib.compress(bytes(raw), level)) + chunk(b"IEND", b""))


def test_image_decoders(ptb, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)      # save_image takes exactly one '.' in the whole path: relative names for the writers below
    rng = np.random.default_rng(5)
    img8 = rng.integers(0, 256, (9, 11, 3)).astype(np.uint8)
    want = img8.astype(np.float32) / 255.0                                  # to_rgb32f
    # compressed png, dynamic + fixed huffman + stored blocks
    for level in (0, 1, 9):
        f = tmp_path / f"a{level}.png"
        f.write_bytes(_png_bytes(img8, level=level))
        assert np.array_equal(ptb.load_image(str(f)), want)
    big = np.tile(img8, (30, 30, 1))                                        # long matches, multiple blocks
    f = tmp_path / "big.png"
    f.write_bytes(_png_bytes(big))
    assert np.array_equal(ptb.load_image(str(f)), big.astype(np.float32) / 255.0)
    img16 = rng.integers(0, 65536, (5, 6, 3)).astype(np.uint16)
    f = tmp_path / "b.png"
    f.write_bytes(_png_bytes(img16, bit_depth=16))
    assert np.array_equal(ptb.load_image(str(f)), img16.astype(np.float32) / 65535.0)
    grey = rng.integers(0, 256, (4, 5, 1)).astype(np.uint8)
    f = tmp_path / "g.png"
    f.write_bytes(_png_bytes(grey, colour_type=0))
    assert np.array_equal(ptb.load_image(str(f)), np.repeat(grey, 3, axis=2).astype(np.float32) / 255.0)
    rgba = rng.integers(0, 256, (4, 5, 4)).astype(np.uint8)
    f = tmp_path / "rgba.png"
    f.write_bytes(_png_bytes(rgba, colour_type=6))
    assert np.array_equal(ptb.load_image(str(f)), rgba[:, :, :3].astype(np.float32) / 255.0)
    # binary / ascii ppm, bmp, pfm; and a round trip through the library's own writers (output crate side)
    f = tmp_path / "c.ppm"
    f.write_bytes(b"P6\n# comment\n11 9\n255\n" + img8.tobytes())
    assert np.array_equal(ptb.load_image(str(f)), want)
    f = tmp_path / "d.ppm"
    f.write_text("P3\n11 9\n255\n" + " ".join(map(str, img8.reshape(-1))) + "\n")
    assert np.array_equal(ptb.load_image(str(f)), want)
    lin = rng.uniform(0, 4, (9, 11, 3)).astype(np.float32)
    f = tmp_path / "e.pfm"
    ptb.save_image(f.name, 11, 9, lin, 2.2)
    assert np.array_equal(ptb.load_image(str(f)), lin)
    for ext in ("bmp", "png", "ppm"):
        f = tmp_path / f"w.{ext}"
        ptb.save_image(f.name, 11, 9, want, 1.0)                            # gamma 1: v * 255.999 as u8
        assert np.array_equal(ptb.load_image(str(f)), np.floor(want * 255.999).astype(np.float32) / 255.0), ext
    with pytest.raises(ptb.PtbError):
        ptb.load_image(str(tmp_path / "missing.png"))
    (tmp_path / "bad.png").write_bytes(_png_bytes(img8)[:60])
    with pytest.raises(ptb.PtbError):
        ptb.load_image(str(tmp_path / "bad.png"))


def test_loader_new_kinds(ptb, tmp_path):
    """loader/src/textures.rs:50-67, materials.rs:77-102: image / perlin textures and trowbridge_reitz load."""
    img = (np.arange(4 * 6 * 3).reshape(4, 6, 3) % 256).astype(np.uint8)
    (tmp_path / "sky.ppm").write_bytes(b"P6\n6 4\n255\n" + img.tobytes())
    text = """camera (
origin 0 -3 0
lookat 0 0 0
vup 0 0 1
fov 40
)
texture env (
type image
filename sky.ppm
)
texture noise (
type perlin
)
texture chk (
type checkered
primary 1 0 0
secondary 0 1 0
)
material rough (
type trowbridge_reitz
texture chk
alpha 0.4
ior 1.5 1.4 1.3
metallic 0.25
)
material marble (
type lambertian
texture noise
)
sky (
texture env
sampler_res 8 4
)
primitive (
type sphere
material rough
centre 0 0 0
radius 1
)
primitive (
type sphere
material marble
centre 2 0 0
)
"""
    s = ptb.load_str(text, str(tmp_path))
    kinds = list(s.textures["kind"])
    assert kinds[:3] == [ptb.TEX_IMAGE, ptb.TEX_PERLIN, ptb.TEX_CHECKERED]
    w, h, words = s.texture_data[0]
    assert (w, h) == (6, 4) and np.array_equal(words.reshape(4, 6, 3), img.astype(np.float32) / 255.0)
    assert s.texture_data[1][2].size == 1024
    m = s.materials[0]
    assert m["kind"] == ptb.MAT_TROWBRIDGE_REITZ and abs(m["param"] - 0.16) < 1e-7      # alpha stored squared
    assert np.allclose(m["ior"], (1.5, 1.4, 1.3)) and m["metallic"] == 0.25
    with pytest.raises(ptb.PtbError) as e:
        ptb.load_str("texture t (\ntype image\n)\n", str(tmp_path))
    assert e.value.code == 6   # MissingRequired("filename")
    with pytest.raises(ptb.PtbError):
        ptb.load_str("texture t (\ntype image\nfilename nope.png\n)\n", str(tmp_path))
