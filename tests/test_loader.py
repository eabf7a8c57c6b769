"""Host-side ingest (host/ssml_loader.cpp) against the reference loader's documented behaviour
(crates/loader/src/*.rs, SURVEY.md appendix A) and the smoke tests it ships
(loader/src/textures.rs:90-117, materials.rs:117-135, primitives.rs:58-90, lib.rs:495-507). No GPU."""
import os

import numpy as np
import pytest


def test_shipped_scenes_parse(ptb, rtweekend1, overshadowed):
    assert len(rtweekend1.spheres) == 2 and len(rtweekend1.triangles) == 0
    assert list(rtweekend1.textures["kind"]) == [ptb.TEX_LERP, ptb.TEX_SOLID, ptb.TEX_SOLID]   # sky, grey, __DEFAULT_TEX
    assert np.allclose(rtweekend1.textures["a"][0], [0.5, 0.7, 1.0]) and np.allclose(rtweekend1.textures["b"][0], 1.0)
    assert list(rtweekend1.materials["kind"]) == [ptb.MAT_LAMBERTIAN, ptb.MAT_LAMBERTIAN]       # ground, __DEFAULT_MAT
    assert rtweekend1.materials["param"][1] == np.float32(0.25) and rtweekend1.materials["texture"][1] == 2
    assert tuple(rtweekend1.sky[0]) == (0, 100, 100)                                             # default sampler_res
    # overshadowed: spheres first, then the 12 aacuboid triangles in the order of meshes.rs:87-100
    assert len(overshadowed.spheres) == 2 and len(overshadowed.triangles) == 12
    assert overshadowed.materials["kind"][1] == ptb.MAT_EMIT and overshadowed.materials["param"][1] == np.float32(1.5)
    t = overshadowed.triangles
    assert np.allclose(t["p"][0], [[-0.5, 0.1, -0.5], [-0.4, 0.1, -0.5], [-0.4, 0.2, -0.5]])
    assert np.allclose(t["n"][0], [[0, 0, -1]] * 3) and np.allclose(t["n"][11], [[0, 0, 1]] * 3)
    assert np.allclose(t["p"][11], [[-0.5, 0.1, -0.4], [-0.4, 0.2, -0.4], [-0.5, 0.2, -0.4]])


def test_loader_smoke_scene_of_the_reference(ptb):
    """crates/loader/src/lib.rs:433-507 (three spheres)."""
    s = ptb.load_str("""camera (
	origin   -5 3 -3
	lookat   0 0.5 0
	vup      0 1 0
	fov      34.0
	aperture 0.0
	focus_dis 10.0
)

texture sky (
	type solid
	colour 0.0
)

sky (
	texture sky
)

texture grey (
	type solid
	colour 0.5
)

texture white (
	type solid
	colour 1.0
)

material ground (
	type lambertian
	texture grey
	albedo 0.5
)

material light (
	type emissive
	texture white
	strength 1.5
)

primitive (
	type sphere
	material ground
	centre 0 -1000 0
	radius 1000
)

primitive (
	type sphere
	material light
	centre 0 0.5 0
	radius 0.5
)

primitive (
	type sphere
	material ground
	centre -0.45 0.15 -0.45
	radius 0.05
)""")
    assert len(s.spheres) == 3 and s.spheres["material"].tolist() == [0, 1, 0]


def test_defaults_and_autocast(ptb):
    s = ptb.load_str("#ver1\ncamera (\n)\nprimitive (\n\ttype sphere\n\tcentre 1\n)\n")
    # camera defaults: origin (3,0,0), lookat 0, vup y, fov 40, focus 10, aspect 16/9 (loader/src/misc.rs:8-15)
    assert np.allclose(s.camera["origin"][0], [3, 0, 0])
    # missing sky -> defaults; unnamed material -> __DEFAULT_MAT (lambertian 0.25 on solid 1.0)
    assert tuple(s.sky[0]) == (0, 100, 100) and len(s.textures) == 1 and len(s.materials) == 1
    assert np.allclose(s.spheres["center"][0], [1, 1, 1]) and s.spheres["radius"][0] == 1.0   # Num1 -> Vec3 autocast
    assert s.materials["kind"][0] == ptb.MAT_LAMBERTIAN and s.materials["param"][0] == np.float32(0.25)
    s = ptb.load_str("camera (\n)\nsky (\n\tsampler_res 0\n)\n")
    assert tuple(s.sky[0])[1:] == (0, 0)
    s = ptb.load_str("camera (\n)\nmaterial m (\n\ttype trowbridge_reitz\n\talpha 0.3\n)\n")
    assert s.materials["kind"][0] == ptb.MAT_TROWBRIDGE_REITZ and np.isclose(s.materials["param"][0], 0.09)  # stored squared
    for kind, key, default in (("reflect", "fuzz", 0.1), ("refract", "eta", 1.5), ("emissive", "strength", 1.5),
                               ("lambertian", "albedo", 0.5)):
        s = ptb.load_str(f"camera (\n)\nmaterial m (\n\ttype {kind}\n)\n")
        assert s.materials["param"][0] == np.float32(default)


@pytest.mark.parametrize("text,code", [
    ("camera (\n\tfov 34.0 \n)\n", 4),                      # trailing blank after a value: line_ending fails -> ParseError
    ("camera (\n\tfov 34.0\n) trailing", 4),                # unparsed trailing input
    ("camera (\n\tfov 34.0)", 4),                           # last key/value line must end in a newline
    ("texture t (\n\ttype solid\n)\n", 6),                  # MissingCamera
    ("camera (\n)\ntexture t (\n\tcolour 1\n)\n", 6),       # MissingRequiredVariantType
    ("camera (\n)\ntexture t (\n\ttype wood\n)\n", 6),      # unknown texture type
    ("camera (\n)\nprimitive (\n\ttype sphere\n)\n", 6),    # sphere without centre
    ("camera (\n)\nprimitive (\n\ttype triangle\n)\n", 8),  # todo!() in the reference
    ("camera (\n)\nmesh (\n\ttype mesh\n)\n", 6),           # mesh without obj
    ("camera (\n)\nmesh (\n\ttype mesh\n\tobj /nonexistent/x.obj\n)\n", 5),
])
def test_rejects_what_the_reference_rejects(ptb, text, code):
    with pytest.raises(ptb.PtbError) as e:
        ptb.load_str(text)
    assert e.value.code == code


def test_duplicate_names_and_last_key_wins(ptb):
    s = ptb.load_str("camera (\n)\ntexture a (\n\ttype solid\n\tcolour 0.1\n\tcolour 0.2\n)\n"
                     "texture a (\n\ttype solid\n\tcolour 0.9\n)\nmaterial m (\n\ttype lambertian\n\ttexture a\n)\n")
    assert np.allclose(s.textures["a"][0], 0.2)           # HashMap: the repeated key keeps the last value
    assert s.materials["texture"][0] == 1                  # the later texture named `a` overwrote the lookup entry


def test_obj_mesh_roundtrip(ptb, tmp_path):
    small = ptb.meshgen.c3_scene(0.01)
    obj = tmp_path / "mesh.obj"
    ptb.meshgen.write_obj(str(obj), small)
    ssml = tmp_path / "scene.ssml"
    ssml.write_text(ptb.meshgen.c3_ssml("mesh.obj"))           # relative path: resolved against the scene file
    s = ptb.load_file(str(ssml))
    assert len(s.triangles) == len(small.triangles)
    assert np.array_equal(s.triangles["p"], small.triangles["p"])
    assert np.array_equal(s.triangles["n"], small.triangles["n"])
    names = {0: ptb.MAT_LAMBERTIAN, 1: ptb.MAT_REFRACT}
    assert all(s.materials["kind"][m] == names[int(k)] for m, k in zip(s.triangles["material"], small.triangles["material"]))
    assert np.array_equal(s.camera, small.camera)


def test_obj_without_normals_is_rejected(ptb, tmp_path):
    (tmp_path / "m.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    with pytest.raises(ptb.PtbError):
        ptb.load_str("camera (\n)\nmesh (\n\ttype mesh\n\tobj m.obj\n)\n", base_dir=str(tmp_path))
    (tmp_path / "q.obj").write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvn 0 0 1\nf 1//1 2//1 3//1 4//1\nf -4//-1 -3//-1 -2//-1\n")
    s = ptb.load_str("camera (\n)\nmesh (\n\ttype mesh\n\tobj q.obj\n)\n", base_dir=str(tmp_path))
    assert len(s.triangles) == 3                                # quad -> fan of 2, plus one negative-index triangle
    assert s.triangles["material"].tolist() == [0, 0, 0]        # no usemtl, no "default" material -> __DEFAULT_MAT


def test_image_save(ptb, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)      # relative names: the one-'.' rule covers the whole path, so a '.' in tmp_path would trip it
    img = np.linspace(0, 1.2, 8 * 4 * 3, dtype=np.float32).reshape(4, 8, 3)
    for ext in ("ppm", "bmp", "png", "pfm"):
        p = tmp_path / f"out.{ext}"
        ptb.save_image(p.name, 8, 4, img, 2.2)
        assert p.stat().st_size > 0
    raw = (tmp_path / "out.ppm").read_bytes()
    px = np.frombuffer(raw[raw.index(b"255\n") + 4:], np.uint8)
    vals = np.power(img.ravel(), np.float32(1 / 2.2)) * np.float32(255.999)
    assert np.array_equal(px, np.clip(vals, 0, 255).astype(np.uint8))     # output/src/lib.rs:92-95
    with pytest.raises(ptb.PtbError):
        ptb.save_image("a.b.png", 8, 4, img)                                # filename must split into exactly two parts
    with pytest.raises(ptb.PtbError):
        ptb.save_image("out.webp", 8, 4, img)


def _read_exr(path):
    """Minimal reader of the OpenEXR 2 scanline layout ("OpenEXR File Layout": magic, version, attributes, offset table,
    per-scanline chunks with the channels in alphabetical order) — enough to check the writer against the specification."""
    import struct
    raw = open(path, "rb").read()
    assert struct.unpack_from("<II", raw, 0) == (20000630, 2)
    pos, attrs = 8, {}
    while raw[pos] != 0:
        e = raw.index(b"\0", pos); name = raw[pos:e].decode(); pos = e + 1
        e = raw.index(b"\0", pos); typ = raw[pos:e].decode(); pos = e + 1
        (size,) = struct.unpack_from("<i", raw, pos); pos += 4
        attrs[name] = (typ, raw[pos:pos + size]); pos += size
    pos += 1
    assert attrs["compression"] == ("compression", b"\0") and attrs["lineOrder"] == ("lineOrder", b"\0")
    x0, y0, x1, y1 = struct.unpack("<4i", attrs["dataWindow"][1])
    w, h = x1 - x0 + 1, y1 - y0 + 1
    chans, c = [], attrs["channels"][1]
    q = 0
    while c[q] != 0:
        e = c.index(b"\0", q); chans.append(c[q:e].decode())
        assert struct.unpack_from("<i", c, e + 1)[0] == 2        # FLOAT
        q = e + 1 + 16
    assert chans == sorted(chans) == ["B", "G", "R"]
    offsets = struct.unpack_from(f"<{h}Q", raw, pos)
    img = np.zeros((h, w, 3), np.float32)
    for y, off in enumerate(offsets):
        yy, size = struct.unpack_from("<ii", raw, off)
        assert yy == y and size == 12 * w
        row = np.frombuffer(raw, np.float32, 3 * w, off + 8).reshape(3, w)
        img[y] = row[::-1].T                                        # B, G, R planes -> RGB pixels
    assert offsets[-1] + 8 + 12 * w == len(raw)
    return img


def test_image_save_every_reference_extension(ptb, tmp_path, monkeypatch):
    """SURVEY.md §8(f) N2 — output/src/lib.rs:89-107: png | jpg | jpeg | tiff | ppm | bmp through the 8-bit gamma mapping,
    exr as linear f32. The files are read back with independent decoders (Pillow; the EXR layout parser above)."""
    from PIL import Image
    monkeypatch.chdir(tmp_path)      # relative names, as in test_image_save
    w, h = 67, 45                                                    # not multiples of the 8 x 8 JPEG block
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([xx / w, yy / h, 0.5 + 0.5 * np.sin(xx / 5.0) * np.cos(yy / 7.0)], -1).astype(np.float32)
    img[5:9, 5:9] = [2.0, 0.0, 1.5]                                  # saturates: Rust `as u8` clamps
    img[0, 0] = [np.nan, -1.0, 0.25]                                 # NaN and negatives -> 0
    want8 = np.clip(np.nan_to_num(np.power(img, np.float32(1 / 2.2)) * np.float32(255.999), nan=0.0), 0, 255).astype(np.uint8)
    for ext in ("png", "tiff", "bmp", "ppm"):
        f = tmp_path / f"o.{ext}"
        ptb.save_image(f.name, w, h, img, 2.2)
        assert np.array_equal(np.asarray(Image.open(f).convert("RGB")), want8), ext
    for ext in ("jpg", "jpeg"):
        f = tmp_path / f"o.{ext}"
        ptb.save_image(f.name, w, h, img, 2.2)
        im = Image.open(f)
        assert im.format == "JPEG" and im.size == (w, h)
        got = np.asarray(im.convert("RGB")).astype(np.float64)
        ours = np.sqrt(np.mean((got - want8) ** 2))
        g = tmp_path / "pil.jpg"                                     # Pillow's own quality-75 4:4:4 encode of the same pixels
        Image.fromarray(want8).save(g, quality=75, subsampling=0)
        theirs = np.sqrt(np.mean((np.asarray(Image.open(g)).astype(np.float64) - want8) ** 2))
        assert ours < 1.25 * theirs + 0.5, (ours, theirs)
    f = tmp_path / "o.exr"
    ptb.save_image(f.name, w, h, img, 2.2)                           # gamma is ignored for exr (lib.rs:98-99)
    back = _read_exr(f)
    assert np.array_equal(back.view(np.uint32), img.view(np.uint32))    # linear f32, bit for bit (NaN included)
