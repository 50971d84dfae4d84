"""Scene ingestion (SURVEY.md §8f-2) and image files (§8f-3): Mitsuba XML -> flat scene, Radiance .hdr, PNG.
CPU only.  The reference importers are src/common/importer/mitsuba.rs + src/pathtracer/importer/mitsuba.rs."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _materials(flat):
    d = flat.desc.contents
    return [d.materials[i] for i in range(d.n_materials)]


def _tex(flat, i):
    return flat.desc.contents.textures[i]


def test_snake_case_matches_heck(host):
    # parameter names go through heck::SnakeCase (common/importer/mitsuba.rs:189, 239, 338)
    want = {"intIOR": "int_ior", "extIOR": "ext_ior", "specularReflectance": "specular_reflectance", "diffuseReflectance": "diffuse_reflectance",
            "uscale": "uscale", "color0": "color0", "alpha": "alpha", "faceNormals": "face_normals", "toWorld": "to_world", "k": "k"}
    for src, dst in want.items():
        assert host.snake_case(src) == dst


def test_cornell_xml_equals_the_transcribed_scene(host):
    """data/cornell-box.xml (fixture with the same numbers) through the XML importer == the hand-transcribed
    build_cornell(): nodes, primitive order, vertices, lights and the camera, bit for bit."""
    a, ca = host.import_scene(os.path.join(GOLDEN, "cornell-box.xml"), res=(512, 512))
    b, cb = host.make_scene(host.SCENE_CORNELL, res=(512, 512))
    assert (a.n_prims, a.n_nodes, a.n_lights) == (36, 59, 2) == (b.n_prims, b.n_nodes, b.n_lights)
    assert np.array_equal(a.nodes(), b.nodes())
    assert np.array_equal(a.prim_vertices(), b.prim_vertices())
    assert bytes(ca) == bytes(cb)
    da, db = a.desc.contents, b.desc.contents
    for i in range(da.n_prims):
        ma, mb = da.materials[da.prim_material[i]], db.materials[db.prim_material[i]]
        assert ma.type == mb.type == host.MAT_MATTE
        assert list(_tex(a, ma.tex[0]).v1) == list(_tex(b, mb.tex[0]).v1)
        assert da.prim_area_light[i] == db.prim_area_light[i]
    la = [da.lights[i] for i in range(2)]
    assert all(l.type == host.LIGHT_AREA for l in la)
    assert list(_tex(a, la[0].ke_tex).v1) == [17.0, 12.0, 4.0]


def test_resolution_only_changes_the_camera(host):
    # -r is the only source of image size and aspect; the XML film size only scales the fov (mitsuba.rs:687-705)
    _, c1 = host.import_scene(os.path.join(GOLDEN, "cornell-box.xml"), res=(640, 480))
    c2 = host.mitsuba_camera(np.array([-1, 0, 0, 0, 0, 1, 0, 1, 0, 0, -1, 6.8, 0, 0, 0, 1], dtype=np.float32), 19.5, 1024, 1024, 640, 480)
    assert (c1.width, c1.height) == (640, 480)
    assert bytes(c1) == bytes(c2)


def test_sunsky_maps_to_an_environment_map(host, tmp_path):
    # importer/mitsuba.rs:400-418: sunsky -> InfiniteAreaLight(env_light_to_world, default .hdr), pushed into both light lists
    sky = host.synth_sky(64, 32, seed=3)
    host.save_hdr(str(tmp_path / "sky.hdr"), sky)
    flat, _ = host.import_scene(os.path.join(GOLDEN, "cornell-box-sunsky.xml"), res=(64, 64), sunsky_hdr=str(tmp_path / "sky.hdr"))
    d = flat.desc.contents
    assert d.n_lights == 3 and d.n_infinite_lights == 1 and d.infinite_lights[0] == 2
    assert d.lights[2].type == host.LIGHT_INFINITE
    e = d.envs[0]
    assert (e.nu, e.nv) == (128, 64)  # distribution at twice the map resolution (light.rs:375-387)
    assert np.allclose(np.array(e.light_to_world).reshape(4, 4), host.mitsuba_env_light_to_world())
    # without a path the seeded synthetic sky stands in (the reference's file does not ship with the repo)
    flat2, _ = host.import_scene(os.path.join(GOLDEN, "cornell-box-sunsky.xml"), res=(64, 64))
    assert flat2.desc.contents.envs[0].nu == 2048


SCENE_ALL = """<?xml version="1.0" encoding="utf-8"?>
<!-- every bsdf / shape / texture kind of common/importer/mitsuba.rs -->
<scene version="0.5.0">
  <sensor type="perspective">
    <float name="fov" value="40"/>
    <transform name="toWorld"><matrix value="-1 0 0 0 0 1 0 1 0 0 -1 8 0 0 0 1"/></transform>
    <film type="ldrfilm"><integer name="width" value="800"/><integer name="height" value="600"/></film>
  </sensor>
  <bsdf type="diffuse" id="white"/>
  <bsdf type="diffuse" id="checker">
    <texture type="checkerboard">
      <rgb name="color0" value="0.1, 0.2, 0.3"/><rgb name="color1" value="0.9, 0.8, 0.7"/>
      <float name="uscale" value="4"/><float name="vscale" value="5"/><float name="uoffset" value="0.25"/><float name="voffset" value="0.5"/>
    </texture>
  </bsdf>
  <bsdf type="diffuse" id="image"><texture type="bitmap"><string name="filename" value="tex.png"/></texture></bsdf>
  <bsdf type="conductor" id="mirror"><string name="material" value="none"/></bsdf>
  <bsdf type="conductor" id="copper"><rgb name="eta" value="0.2, 0.92, 1.1"/><rgb name="k" value="3.9, 2.45, 2.14"/></bsdf>
  <bsdf type="roughconductor" id="rough">
    <float name="alpha" value="0.15"/><rgb name="eta" value="0.2, 0.92, 1.1"/><rgb name="k" value="3.9, 2.45, 2.14"/>
    <rgb name="specularReflectance" value="0.5, 0.6, 0.7"/>
  </bsdf>
  <bsdf type="dielectric" id="glass"><float name="intIOR" value="1.5"/><float name="extIOR" value="1"/></bsdf>
  <bsdf type="plastic" id="plastic"><float name="intIOR" value="1.5"/><rgb name="diffuseReflectance" value="0.3, 0.4, 0.5"/></bsdf>
  <bsdf type="twosided" id="roughplastic">
    <bsdf type="roughplastic"><float name="intIOR" value="1.9"/><float name="alpha" value="0.2"/></bsdf>
  </bsdf>
  <shape type="rectangle"><transform name="toWorld"><matrix value="4 0 0 0 0 0 4 0 0 -4 0 0 0 0 0 1"/></transform><ref id="checker"/></shape>
  <shape type="cube"><transform name="toWorld"><matrix value="0.5 0 0 -2 0 0.5 0 0.5 0 0 0.5 0 0 0 0 1"/></transform><ref id="copper"/></shape>
  <shape type="sphere"><point name="center" x="1" y="1" z="0.5"/><float name="radius" value="0.75"/><ref id="glass"/></shape>
  <shape type="obj">
    <string name="filename" value="tri.obj"/>
    <transform name="toWorld"><matrix value="1 0 0 0 0 1 0 2 0 0 1 0 0 0 0 1"/></transform>
    <bsdf type="diffuse"><rgb name="reflectance" value="0.2, 0.3, 0.4"/></bsdf>
    <emitter type="area"><rgb name="radiance" value="5, 6, 7"/></emitter>
  </shape>
  <emitter type="point"/>
</scene>
"""


def test_every_bsdf_shape_and_texture_kind(host, tmp_path):
    (tmp_path / "all.xml").write_text(SCENE_ALL)
    (tmp_path / "tri.obj").write_text("o quad\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvn 0 0 1\nvn 0 0 1\nvn 0 0 1\nvn 0 0 1\n"
                                     "vt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\nf 1/1/1 2/2/2 3/3/3\nf 1/1/1 3/3/3 4/4/4\n")
    rng = np.random.default_rng(5)
    tex = rng.integers(0, 256, (8, 16, 3), dtype=np.uint8)
    host.save_png(str(tmp_path / "tex.png"), tex)
    flat, cam = host.import_scene(str(tmp_path / "all.xml"), res=(320, 240))
    d = flat.desc.contents
    assert (cam.width, cam.height) == (320, 240)
    mats = _materials(flat)
    by_type = {}
    for m in mats:
        by_type.setdefault(m.type, []).append(m)
    # document order: white, checker, image, mirror, copper, rough, glass, plastic, roughplastic, + the embedded diffuse
    assert [m.type for m in mats] == [host.MAT_MATTE, host.MAT_MATTE, host.MAT_MATTE, host.MAT_MIRROR, host.MAT_METAL, host.MAT_METAL,
                                      host.MAT_GLASS, host.MAT_SUBSTRATE, host.MAT_SUBSTRATE, host.MAT_MATTE]
    assert list(_tex(flat, mats[0].tex[0]).v1) == [1.0, 1.0, 1.0]  # default_rgb_one
    ck = _tex(flat, mats[1].tex[0])
    assert ck.type == host.TEX_CHECKER and np.allclose(list(ck.v1), [0.1, 0.2, 0.3]) and (ck.su, ck.sv, ck.du, ck.dv) == (4.0, 5.0, 0.25, 0.5)
    im = _tex(flat, mats[2].tex[0])
    assert im.type == host.TEX_IMAGE and (im.su, im.sv) == (1.0, -1.0)  # UVMap::new(1., -1., 0., 0.), importer/mitsuba.rs:56
    mm = d.mipmaps[im.mip]
    assert (mm.width[0], mm.height[0]) == (16, 8)
    lvl0 = np.ctypeslib.as_array(d.texels, shape=(d.n_texels,))[mm.level_offset[0]: mm.level_offset[0] + 16 * 8 * 3].reshape(8, 16, 3)
    v = tex.astype(np.float32) / np.float32(255)
    want = np.where(v <= 0.04045, v / np.float32(12.92), ((v + np.float32(0.055)) / np.float32(1.055)) ** np.float32(2.4))  # math.rs:141-147
    assert np.allclose(lvl0, want, rtol=2e-6, atol=1e-7)
    copper, rough = mats[4], mats[5]
    assert _tex(flat, copper.tex[3]).v1[0] == np.float32(0.001) and copper.remap_roughness == 0
    assert np.allclose(list(_tex(flat, copper.tex[0]).v1), [0.2, 0.92, 1.1]) and np.allclose(list(_tex(flat, copper.tex[1]).v1), [3.9, 2.45, 2.14])
    assert list(_tex(flat, copper.tex[2]).v1) == [1.0, 1.0, 1.0]
    assert _tex(flat, rough.tex[3]).v1[0] == np.float32(0.15) and np.allclose(list(_tex(flat, rough.tex[2]).v1), [0.5, 0.6, 0.7])
    glass = mats[6]
    assert _tex(flat, glass.tex[2]).v1[0] == 1.5
    plastic, rplastic = mats[7], mats[8]
    r0 = np.float32((np.float32(1.5) - 1) ** 2) / np.float32((np.float32(1.5) + 1) ** 2)  # schlick_r0_from_eta
    assert _tex(flat, plastic.tex[1]).v1[0] == r0 and _tex(flat, plastic.tex[2]).v1[0] == np.float32(0.001)
    assert np.allclose(list(_tex(flat, plastic.tex[0]).v1), [0.3, 0.4, 0.5])
    assert _tex(flat, rplastic.tex[2]).v1[0] == np.float32(0.2) and list(_tex(flat, rplastic.tex[0]).v1) == [1.0, 1.0, 1.0]
    # shapes: rectangle 2 + cube 12 + sphere (10 x 10 lat-long: 10 + 10 fans, 8 x 10 quads) + obj 2 triangles
    n_sphere = d.n_prims - 2 - 12 - 2
    assert n_sphere == 10 * 2 + 8 * 10 * 2
    assert d.n_lights == 2  # one DiffuseAreaLight per emissive triangle; the standalone point emitter is ignored
    light_tris = flat.prim_vertices()[[d.lights[i].prim for i in range(2)]]
    assert np.allclose(light_tris[..., 1].min(), 2.0) and np.allclose(light_tris[..., 1].max(), 3.0)  # obj translated by +2 in y
    pv = flat.prim_vertices()
    sphere_mat = [i for i in range(d.n_prims) if d.materials[d.prim_material[i]].type == host.MAT_GLASS]
    c = pv[sphere_mat].reshape(-1, 3)
    assert len(sphere_mat) == n_sphere
    assert np.allclose(np.linalg.norm(c - np.array([1, 1, 0.5], dtype=np.float32), axis=1), 0.75, atol=1e-5)


def test_importer_errors_mirror_the_reference_panics(host, tmp_path):
    (tmp_path / "a.txt").write_text("x")
    host.save_png(str(tmp_path / "tex.png"), np.zeros((2, 2, 3), dtype=np.uint8))
    (tmp_path / "tri.obj").write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nvn 0 0 1\nvn 0 0 1\nvn 0 0 1\nf 1//1 2//2 3//3\n")
    with pytest.raises(RuntimeError, match="unsupported format"):
        host.import_scene(str(tmp_path / "a.txt"))
    (tmp_path / "noref.xml").write_text(SCENE_ALL.replace('<ref id="copper"/>', ""))
    with pytest.raises(RuntimeError, match="either ref exists or embedded bsdf exists"):
        host.import_scene(str(tmp_path / "noref.xml"))
    (tmp_path / "badmat.xml").write_text(SCENE_ALL.replace('value="none"', 'value="Au"'))
    with pytest.raises(RuntimeError, match="other material values not supported"):
        host.import_scene(str(tmp_path / "badmat.xml"))
    (tmp_path / "broken.xml").write_text("<scene><sensor></scene>")
    with pytest.raises(RuntimeError, match="XML"):
        host.import_scene(str(tmp_path / "broken.xml"))


# ---- image files ---------------------------------------------------------------------------------------
def test_hdr_decoder_known_answers(host, tmp_path):
    """Rgbe8Pixel::to_hdr (image 0.23.14): e == 0 -> 0, else c * 2^(e - 136).  Flat, new-style RLE and old-style runs."""
    head = b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y 2 +X 8\n"
    # scanline 0: new-style RLE (2, 2, 0, 8): R = run of 8 x 128, G = literal 8 bytes, B = run 5 x 64 + literal 3, E = run 8 x 129
    row0 = bytes([2, 2, 0, 8]) + bytes([128 + 8, 128]) + bytes([8, 1, 2, 3, 4, 5, 6, 7, 8]) + bytes([128 + 5, 64, 3, 9, 10, 11]) + bytes([128 + 8, 129])
    # scanline 1: flat pixel, old-style repeat x3, a pixel with zero exponent, three more flat pixels
    row1 = bytes([200, 100, 50, 130]) + bytes([1, 1, 1, 3]) + bytes([255, 255, 255, 0]) + bytes([10, 20, 30, 120]) * 3
    (tmp_path / "k.hdr").write_bytes(head + row0 + row1)
    img = host.load_hdr(str(tmp_path / "k.hdr"))
    assert img.shape == (2, 8, 3)
    s = np.float32(2.0) ** np.float32(129 - 136)
    assert np.array_equal(img[0, :, 0], np.full(8, 128 * s, dtype=np.float32))
    assert np.array_equal(img[0, :, 1], np.arange(1, 9, dtype=np.float32) * s)
    assert np.array_equal(img[0, :, 2], np.array([64] * 5 + [9, 10, 11], dtype=np.float32) * s)
    s1 = np.float32(2.0) ** np.float32(130 - 136)
    assert np.array_equal(img[1, :4], np.tile(np.array([200, 100, 50], dtype=np.float32) * s1, (4, 1)))
    assert np.array_equal(img[1, 4], np.zeros(3, dtype=np.float32))
    assert np.array_equal(img[1, 5], np.array([10, 20, 30], dtype=np.float32) * np.float32(2.0) ** np.float32(120 - 136))


def test_hdr_round_trip(host, tmp_path):
    rng = np.random.default_rng(1)
    x = (rng.random((20, 33, 3)) * 40).astype(np.float32)
    x[3, 4] = 0
    host.save_hdr(str(tmp_path / "x.hdr"), x)
    y = host.load_hdr(str(tmp_path / "x.hdr"))
    assert y.shape == x.shape and np.all(y[3, 4] == 0)
    assert np.abs(y - x).max() <= x.max(axis=2, keepdims=True).max() / 128  # 8-bit mantissa shared exponent


def test_hdr_decoder_on_the_reference_map_matches_opencv(host):
    """The reference's own environment map (data/abandoned_tank_farm_04_1k.hdr), committed as tests/golden's fixture."""
    cv2 = pytest.importorskip("cv2")
    img = host.load_hdr(host.TANK_FARM_HDR)
    ref = cv2.imread(host.TANK_FARM_HDR, cv2.IMREAD_UNCHANGED)[..., ::-1]
    assert img.shape == (512, 1024, 3) and np.array_equal(img, ref)


def test_png_round_trip_and_pil_interop(host, tmp_path):
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(2)
    for c in (1, 2, 3, 4):
        a = rng.integers(0, 256, (37, 53, c), dtype=np.uint8)
        p = str(tmp_path / f"a{c}.png")
        host.save_png(p, a)
        assert np.array_equal(host.load_png(p), a)
        assert np.array_equal(np.asarray(Image.open(p)).reshape(37, 53, c), a)
    grad = np.linspace(0, 255, 64 * 64 * 3).reshape(64, 64, 3).astype(np.uint8)  # PIL picks adaptive row filters here
    Image.fromarray(grad).save(str(tmp_path / "p.png"), optimize=True)
    assert np.array_equal(host.load_png(str(tmp_path / "p.png")), grad)
    Image.fromarray(grad).convert("P", colors=64).save(str(tmp_path / "pal.png"))
    assert np.array_equal(host.load_png(str(tmp_path / "pal.png")), np.asarray(Image.open(str(tmp_path / "pal.png")).convert("RGB")))
    (tmp_path / "bad.png").write_bytes(b"\x89PNG\r\n\x1a\nxxxx")
    with pytest.raises(RuntimeError):
        host.load_png(str(tmp_path / "bad.png"))


# ---- tev display-server messages (src/headless.rs:14-178) -------------------------------------------------
def test_tev_create_image_message(host):
    """The reference's own test (headless.rs:253-288) restated: length prefix, header 4, name, focus, resolution."""
    import struct

    msg = host.tev_create_image(1920, 1080, "render")
    assert struct.unpack_from("<I", msg, 0)[0] == len(msg)
    assert msg[4] == 4 and msg[5] == 1
    assert msg[6:13] == b"render\0"
    assert struct.unpack_from("<iii", msg, 13) == (1920, 1080, 3)
    assert msg[25:] == b"r\0g\0b\0"


def test_tev_update_image_tiles(host):
    import struct

    h, w = 130, 250
    img = np.arange(h * w * 3, dtype=np.float32).reshape(h, w, 3)
    blob = host.tev_update_image(img, "render")
    off, seen = 0, []
    while off < len(blob):
        (n,) = struct.unpack_from("<I", blob, off)
        m = blob[off: off + n]
        assert m[4] == 3 and m[5] == 1 and m[6:13] == b"render\0"
        ch = m[13:14].decode()
        x, y, cw, chh = struct.unpack_from("<iiii", m, 15)
        data = np.frombuffer(m, dtype="<f4", offset=31).reshape(chh, cw)
        assert np.array_equal(data, img[y: y + chh, x: x + cw, "rgb".index(ch)])
        seen.append((ch, x, y, cw, chh))
        off += n
    # per channel: x-major over 100-pixel steps, like (0..w).step_by(100) x (0..h).step_by(100)
    assert seen[:6] == [("r", 0, 0, 100, 100), ("r", 0, 100, 100, 30), ("r", 100, 0, 100, 100), ("r", 100, 100, 100, 30),
                        ("r", 200, 0, 50, 100), ("r", 200, 100, 50, 30)]
    assert [s[0] for s in seen] == ["r"] * 6 + ["g"] * 6 + ["b"] * 6


def test_corrupted_scene_files_raise_or_load(host, tmp_path):
    """Scene files are untrusted input: random edits of the Cornell XML and of a small glTF document must either import
    or raise (the reference panics); the XML / JSON readers and both importers never read out of bounds."""
    import base64
    import json

    rng = np.random.default_rng(5)

    def mutate(data, digits_only=False):
        m = bytearray(data)
        for _ in range(int(rng.integers(1, 6))):
            k = int(rng.integers(0, len(m)))
            op = int(rng.integers(0, 3))
            if op == 0:
                m[k] = int(rng.integers(32, 127))
            elif op == 1:
                del m[k:k + int(rng.integers(1, 20))]
            else:
                m[k:k] = bytes(rng.integers(48 if digits_only else 32, 58 if digits_only else 127, int(rng.integers(1, 8)), dtype=np.uint8))
        return bytes(m)

    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    blob = pos.tobytes() + np.array([0, 1, 2, 0], dtype=np.uint16).tobytes()
    doc = {"asset": {"version": "2.0"}, "scene": 0, "scenes": [{"nodes": [0]}], "nodes": [{"mesh": 0, "translation": [0, 0, -3]}],
           "meshes": [{"primitives": [{"attributes": {"POSITION": 0}, "indices": 1, "material": 0}]}],
           "materials": [{"pbrMetallicRoughness": {"baseColorFactor": [0.8, 0.5, 0.2, 1], "metallicFactor": 0.1}, "emissiveFactor": [1, 1, 1]}],
           "buffers": [{"byteLength": len(blob), "uri": "data:application/octet-stream;base64," + base64.b64encode(blob).decode()}],
           "bufferViews": [{"buffer": 0, "byteOffset": 0, "byteLength": 36}, {"buffer": 0, "byteOffset": 36, "byteLength": 6}],
           "accessors": [{"bufferView": 0, "componentType": 5126, "count": 3, "type": "VEC3", "min": [0, 0, 0], "max": [1, 1, 0]},
                         {"bufferView": 1, "componentType": 5123, "count": 3, "type": "SCALAR"}]}
    sources = {"m.xml": (open(os.path.join(GOLDEN, "cornell-box.xml"), "rb").read(), False), "m.gltf": (json.dumps(doc).encode(), True)}
    for name, (data, digits) in sources.items():
        host.import_scene(_write(tmp_path / name, data), res=(32, 32))  # the unmodified file loads
        outcomes = {"ok": 0, "error": 0}
        for _ in range(120):
            try:
                host.import_scene(_write(tmp_path / name, mutate(data, digits)), res=(32, 32))
                outcomes["ok"] += 1
            except RuntimeError:
                outcomes["error"] += 1
        assert outcomes["error"] > 30, (name, outcomes)


def _write(path, data):
    path.write_bytes(data)
    return str(path)
