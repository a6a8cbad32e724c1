"""RTXPT .scene.json loading (rtxpt_b200_load_scene_json): models instanced through the graph with translation / rotation / euler / scaling,
lights, cameras, environment light and settings — against the same scene assembled with the numpy table builder.  CPU only."""
import gzip
import json
import os
import numpy as np
import pytest
import gltf_export

ASSETS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_assets.json.gz")


def _quat_matrix(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]], np.float64)


def _xf(t=(0, 0, 0), q=(0, 0, 0, 1), s=(1, 1, 1)):
    m = np.eye(4); m[:3, :3] = _quat_matrix(q) @ np.diag(s); m[:3, 3] = t; return m


def test_scene_json_instancing_lights_cameras(product, oracle, tmp_path):
    from rtxpt_b200 import scenes, structs as S
    from rtxpt_b200.scene_builder import SceneBuilder, Material
    from rtxpt_b200.scenes import _quad, _box, _merge
    media = tmp_path / "media"; (media / "Models" / "room").mkdir(parents=True); (media / "Models" / "crate").mkdir(parents=True); (media / "Materials").mkdir()
    # two models: the Cornell box and a crate that the scene instances three times
    room = scenes.cornell_builder()
    gltf_export.export(room, str(media / "Models" / "room" / "room.gltf"))
    crate = SceneBuilder(); cm = crate.add_material(Material(base_color=(0.6, 0.4, 0.2), roughness=0.7))
    crate.add_mesh([_merge(_box([(-0.25, 0, -0.25), (0.25, 0, -0.25), (0.25, 0, 0.25), (-0.25, 0, 0.25)], 0.5, cm), cm)]); crate.add_instance(0)
    gltf_export.export(crate, str(media / "Models" / "crate" / "crate.glb"), glb=True)
    (media / "Materials" / "crate.mat0.material.json").write_text(json.dumps({"Roughness": 0.25, "Metalness": 1.0, "BaseOrDiffuseColor": [0.9, 0.8, 0.7]}))
    h = np.sqrt(0.5)
    scene_json = {
        "models": ["Models/room/room.gltf", "Models\\crate\\crate.glb"],
        "graph": [
            {"name": "Room", "model": 0},
            {"name": "CrateA", "model": 1, "translation": [1.0, 0.0, 1.5]},
            {"name": "Group", "translation": [3.0, 0.0, 3.0], "scaling": 2.0, "children": [
                {"name": "CrateB", "model": 1, "rotation": [0, h, 0, h]},
                {"name": "CrateC", "model": 1, "translation": [0.5, 0.25, 0.0], "euler": [0.0, 1.23, 0.0], "scaling": [1.0, 0.5, 1.0]},
                {"name": "BadRotation", "model": 1, "translation": [-0.5, 0, 0], "rotation": [0.7071068, 0, 0.7071068]}]},          # 3 elements: Donut keeps the identity
            {"name": "Lights", "children": [
                {"name": "Sky", "type": "EnvironmentLight", "radianceScale": [1, 2, 3], "rotation": [0.25], "path": "EnvironmentMaps\\sky_cube.dds"},
                {"name": "Sun", "type": "DirectionalLight", "color": [1, 1, 1], "irradiance": 3.0},
                {"name": "Bulb", "type": "PointLight", "translation": [2.0, 4.0, 2.0], "color": [1.0, 0.9, 0.8], "intensity": 25.0, "radius": 0.15},
                {"name": "Spot", "type": "SpotLight", "translation": [4.0, 5.0, 1.0], "euler": [-1.5707963267948966, 0, 0], "color": [0.5, 0.6, 1.0], "intensity": 40.0, "radius": 0.05,
                 "innerAngle": 15.0, "outerAngle": 35.0}]},
            {"name": "Cameras", "children": [
                {"name": "Default", "type": "PerspectiveCameraEx", "translation": [2.78, 2.73, -8.0], "rotation": [0, 1, 0, 0], "verticalFov": 0.66, "zNear": 0.1, "exposureValue": -2.0}]},
            {"name": "SampleSettings", "type": "SampleSettings", "realtimeMode": False, "maxBounces": 12, "maxDiffuseBounces": 3, "realtimeFireflyFilter": 0.15, "startingCamera": "Default"}]}
    path = media / "demo.scene.json"; path.write_text(json.dumps(scene_json, indent=1))
    g = product.GltfScene(str(path))
    # the same scene with the table builder: room instance + 4 crate instances with the composed transforms
    b = scenes.cornell_builder()
    bm = b.add_material(Material(base_color=(0.9, 0.8, 0.7), roughness=0.25, metalness=1.0))
    mesh = b.add_mesh([_merge(_box([(-0.25, 0, -0.25), (0.25, 0, -0.25), (0.25, 0, 0.25), (-0.25, 0, 0.25)], 0.5, bm), bm)])
    group = _xf((3, 0, 3), s=(2, 2, 2))
    ce, se = np.cos(0.5 * 1.23), np.sin(0.5 * 1.23)
    for m in (_xf((1.0, 0.0, 1.5)), group @ _xf(q=(0, h, 0, h)), group @ _xf((0.5, 0.25, 0.0), q=(0, se, 0, ce), s=(1.0, 0.5, 1.0)), group @ _xf((-0.5, 0, 0))):
        b.add_instance(mesh, m[:3, :])
    ref = b.build()
    assert g.desc.instanceCount == ref.desc.instanceCount == 7 and g.triangle_count == ref.triangle_count == 36 + 4 * 12
    for i in range(7):
        a, r = np.array(g.desc.instances[i].transform[:]), np.array(ref.desc.instances[i].transform[:])
        assert np.allclose(a, r, rtol=1e-6, atol=1e-6), (i, a, r)
    # the crate's material came from Materials/crate.mat0.material.json (metal, roughness 0.25); it is the model's material 0, after the room's 4 + default
    crate_mat = g.desc.materials[g.desc.geometries[g.desc.instances[3].firstGeometryIndex].materialIndex]
    assert abs(crate_mat.Roughness - 0.25) < 1e-7 and crate_mat.Metalness == 1.0
    # lights: point + spot (the directional one is counted, not listed), spot axis = -Z of a node pitched -90 degrees about x = straight down
    assert g.desc.lightCount == 2 and g.info.directionalLightCount == 1
    bulb, spot = g.desc.lights[0], g.desc.lights[1]
    assert bulb.type == S.LIGHT_POINT and np.allclose(bulb.position[:], (2, 4, 2)) and abs(bulb.radius - 0.15) < 1e-7 and abs(bulb.intensity - 25.0) < 1e-6
    assert spot.type == S.LIGHT_SPOT and np.allclose(spot.direction[:], (0, -1, 0), atol=1e-6) and (spot.innerAngle, spot.outerAngle) == (15.0, 35.0)
    # camera: rotation (0,1,0,0) = 180 degrees about y: looks down +z from (2.78, 2.73, -8)
    cam = g.cameras[0]
    assert np.allclose(cam.position[:], (2.78, 2.73, -8.0)) and np.allclose(cam.direction[:], (0, 0, 1), atol=1e-6) and np.allclose(cam.up[:], (0, 1, 0), atol=1e-6) and abs(cam.yfov - 0.66) < 1e-7
    info = g.info
    assert info.environmentMapPath.decode() == "EnvironmentMaps/sky_cube.dds" and list(info.environmentRadianceScale) == [1.0, 2.0, 3.0] and abs(info.environmentRotation - 0.25) < 1e-7
    assert info.hasSampleSettings and not info.realtimeMode and (info.maxBounces, info.maxDiffuseBounces) == (12, 3) and info.startingCamera.decode() == "Default" and info.modelCount == 2
    # and the oracle renders both descriptions to the same image
    from rtxpt_b200 import scene_builder as sb
    c = sb.bridge_camera(48, 48, tuple(cam.position[:]), tuple(cam.direction[:]), tuple(cam.up[:]), cam.yfov)
    consts = sb.make_constants(48, 48, c, bounce_count=2, diffuse_bounce_count=2)
    o1 = oracle.Oracle(g); o1.set_constants(consts); a = o1.render(0, 2)[0]; o1.close()
    b2 = scenes.cornell_builder()      # reference scene needs the same analytic lights for the comparison
    bm2 = b2.add_material(Material(base_color=(0.9, 0.8, 0.7), roughness=0.25, metalness=1.0)); mesh2 = b2.add_mesh([_merge(_box([(-0.25, 0, -0.25), (0.25, 0, -0.25), (0.25, 0, 0.25), (-0.25, 0, 0.25)], 0.5, bm2), bm2)])
    for i in range(3, 7): b2.add_instance(mesh2, np.array(g.desc.instances[i].transform[:], np.float32).reshape(3, 4))
    b2.add_point_light((2.0, 4.0, 2.0), (1.0, 0.9, 0.8), 25.0, 0.15); b2.add_spot_light((4.0, 5.0, 1.0), tuple(spot.direction[:]), (0.5, 0.6, 1.0), 40.0, 0.05, 15.0, 35.0)
    r2 = b2.build(); o2 = oracle.Oracle(r2); o2.set_constants(consts); bimg = o2.render(0, 2)[0]; o2.close()
    assert np.abs(a - bimg).max() <= 2e-3 * max(1.0, float(bimg.max()))
    g.close()


def test_scene_json_errors(product, tmp_path):
    p = tmp_path / "x.scene.json"; p.write_text(json.dumps({"models": ["Models/missing.gltf"], "graph": [{"model": 0}]}))
    with pytest.raises(product.RtxptError, match="cannot open"):
        product.GltfScene(str(p))
    p.write_text(json.dumps({"models": [], "graph": [{"name": "n", "model": 3}]}))
    with pytest.raises(product.RtxptError, match="not in the model array"):
        product.GltfScene(str(p))


def test_reference_scene_files_parse_up_to_their_lfs_stubs(product, tmp_path):
    """Every .scene.json the reference ships is read up to the point where its models (git-LFS pointer stubs in the reference checkout) would be parsed.
    The scene files and the stubs they name are laid out again under tmp_path from tests/golden/reference_assets.json.gz.  The expected messages there
    (scene_errors) were recorded from this project's own loader on the reference's Assets tree, not from the reference: they pin the loader's current
    wording as a regression check, and a deliberate rewording of a loader error means regenerating them (tests/golden/make_asset_golden.py)."""
    with gzip.open(ASSETS_GOLDEN, "rt", encoding="utf-8") as f:
        golden = json.load(f)
    for name, text in list(golden["scenes"].items()) + list(golden["models"].items()):
        p = tmp_path / name; p.parent.mkdir(parents=True, exist_ok=True); p.write_text(text, encoding="utf-8")
    files = sorted(golden["scenes"])
    assert len(files) >= 8
    for f in files:
        with pytest.raises(product.RtxptError) as e:
            product.GltfScene(str(tmp_path / f))
        assert "JSON" in str(e.value) or "cannot open" in str(e.value), (f, str(e.value))          # the stub is not JSON / the file is absent; never a crash
        assert str(e.value) == golden["scene_errors"][f].replace("{assets}", str(tmp_path)), (f, str(e.value))
