"""RTXPT .material.json -> PTMaterialData (rtxpt_b200/csrc/material_json.cpp) against an independent Python restatement of PTMaterial::Read +
FillData (Rtxpt/Materials/MaterialsBaker.cpp:160-245, :516-591, defaults MaterialsBaker.h:134-201) — on synthetic files and on every
material file the reference ships (Assets/Materials, 504 files incl. the 254 Bistro materials, stored in tests/golden/reference_assets.json.gz).  CPU only."""
import ctypes as C
import gzip
import json
import os
import numpy as np
import pytest

ASSETS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_assets.json.gz")


def fill_data(j):
    """Independent restatement: returns (MaterialData, info dict)."""
    from rtxpt_b200 import structs as S
    f = np.float32
    g = lambda k, d: j.get(k, d)
    d = S.MaterialData()
    enable_tr = bool(g("EnableTransmission", False))
    flags = 0
    if g("UseSpecularGlossModel", False): flags |= S.MATFLAG_UseSpecularGlossModel
    if g("MetalnessInRedChannel", False): flags |= S.MATFLAG_MetalnessInRedChannel
    if g("ThinSurface", False) or not enable_tr: flags |= S.MATFLAG_ThinSurface
    if g("PSDExclude", True): flags |= S.MATFLAG_PSDExclude
    blk = int(g("PSDBlockMotionVectorsAtSurfaceType", 0))
    if blk % 2: flags |= 1 << 13
    if blk // 2: flags |= 1 << 14
    if g("EnableAsAnalyticLightProxy", False): flags |= S.MATFLAG_EnableAsAnalyticLightProxy
    if g("IgnoreMeshTangentSpace", False): flags |= S.MATFLAG_IgnoreMeshTangentSpace
    flags |= min(int(g("NestedPriority", 14)), 14) << 28
    flags |= min(max(int(g("PSDDominantDeltaLobe", -1)) + 1, 0), 7) << 24
    d.Flags = flags
    d.BaseOrDiffuseColor[:] = [f(x) for x in g("BaseOrDiffuseColor", [1, 1, 1])]
    d.SpecularColor[:] = [f(x) for x in g("SpecularColor", [0, 0, 0])]
    ei = f(g("EmissiveIntensity", 1.0))
    d.EmissiveColor[:] = [f(x) * ei for x in g("EmissiveColor", [0, 0, 0])]
    d.Roughness, d.Metalness, d.NormalTextureScale = f(g("Roughness", 0.0)), f(g("Metalness", 0.0)), f(g("NormalTextureScale", 1.0))
    d.TransmissionFactor = f(g("TransmissionFactor", 0.0)) if enable_tr else 0.0
    d.DiffuseTransmissionFactor = f(g("DiffuseTransmissionFactor", 0.0)) if enable_tr else 0.0
    d.Opacity, d.AlphaCutoff, d.IoR = f(g("Opacity", 1.0)), f(g("AlphaCutoff", 0.5)), f(g("IoR", 1.5))
    d.VolumeAttenuationColor[:] = [f(x) for x in g("VolumeAttenuationColor", [1, 1, 1])]
    d.VolumeAttenuationDistance = f(min(g("VolumeAttenuationDistance", 3.4028234663852886e+38), 3.4028234663852886e+38))
    d.ShadowNoLFadeout = f(min(max(g("ShadowNoLFadeout", 0.0), 0.0), 0.25))
    for k in ("BaseOrDiffuseTextureIndex", "MetalRoughOrSpecularTextureIndex", "EmissiveTextureIndex", "NormalTextureIndex", "OcclusionTextureIndex", "TransmissionTextureIndex"):
        setattr(d, k, 0xFFFFFFFF)
    d._padding0 = 42; d._padding1 = 42.0
    tex = []
    for key, en in (("BaseTexture", "EnableBaseTexture"), ("OcclusionRoughnessMetallicTexture", "EnableOcclusionRoughnessMetallicTexture"), ("NormalTexture", "EnableNormalTexture"),
                    ("EmissiveTexture", "EnableEmissiveTexture"), ("TransmissionTexture", "EnableTransmissionTexture")):
        t = j.get(key) or {}
        path = t.get("path", "").replace("\\", "/")
        tex.append((bool(g(en, True)) and path != "" and (key != "TransmissionTexture" or enable_tr), bool(t.get("sRGB", False)), path))
    return d, dict(alpha=bool(g("EnableAlphaTesting", False)), nee=bool(g("ExcludeFromNEE", False)), skip=bool(g("SkipRender", False)), tr=enable_tr, tex=tex)


def check(product, text):
    info = product.parse_material_json(text)
    ref, meta = fill_data(json.loads(text))
    assert bytes(info.data) == bytes(ref), [(n, getattr(info.data, n), getattr(ref, n)) for n, _ in type(ref)._fields_ if bytes(np.ctypeslib.as_array(getattr(info.data, n)) if hasattr(getattr(ref, n), '__len__') else b'') != b'' or getattr(info.data, n) != getattr(ref, n)][:4]
    assert (bool(info.enableAlphaTesting), bool(info.excludeFromNEE), bool(info.skipRender), bool(info.enableTransmission)) == (meta["alpha"], meta["nee"], meta["skip"], meta["tr"])
    for t in range(5):
        en, srgb, path = meta["tex"][t]
        assert bool(info.textureEnabled[t]) == en and bool(info.textureSRGB[t]) == srgb and info.texturePath[t].value.decode() == path[:259]


def test_material_json_synthetic(product):
    check(product, "{}")                                    # every default
    check(product, json.dumps({"BaseOrDiffuseColor": [0.2, 0.4, 0.6], "Roughness": 0.19, "Metalness": 1.0, "EmissiveColor": [1.0, 0.5, 0.25], "EmissiveIntensity": 12.5,
                               "EnableTransmission": True, "TransmissionFactor": 0.9, "DiffuseTransmissionFactor": 0.1, "ThinSurface": False, "IoR": 1.33, "NestedPriority": 3,
                               "VolumeAttenuationColor": [0.9, 0.95, 1.0], "VolumeAttenuationDistance": 2.0, "PSDExclude": False, "PSDDominantDeltaLobe": 1,
                               "PSDBlockMotionVectorsAtSurfaceType": 3, "ShadowNoLFadeout": 0.4, "EnableAlphaTesting": True, "AlphaCutoff": 0.33, "ExcludeFromNEE": True,
                               "BaseTexture": {"path": "Models\\\\X\\\\a_diff.dds", "sRGB": True, "NormalMap": False}, "EnableBaseTexture": True,
                               "TransmissionTexture": {"path": "t.png", "sRGB": False}, "NormalTexture": {"path": "n.png", "NormalMap": True}, "EnableNormalTexture": False}))
    check(product, json.dumps({"EnableTransmission": False, "TransmissionFactor": 0.7, "TransmissionTexture": {"path": "t.png"}, "UseSpecularGlossModel": True, "SpecularColor": [1, 0.9, 0.8],
                               "MetalnessInRedChannel": True, "EnableAsAnalyticLightProxy": True, "IgnoreMeshTangentSpace": True, "NestedPriority": 99, "SkipRender": True}))
    with pytest.raises(product.RtxptError):
        product.parse_material_json("[1, 2")


def test_material_json_on_reference_assets(product):
    with gzip.open(ASSETS_GOLDEN, "rt", encoding="utf-8") as f:
        files = json.load(f)["materials"]
    assert len(files) > 400
    emissive = transmissive = alpha = 0
    for text in files.values():
        check(product, text)
        j = json.loads(text)
        emissive += any(c > 0 for c in j.get("EmissiveColor", [0])); transmissive += bool(j.get("EnableTransmission")); alpha += bool(j.get("EnableAlphaTesting"))
    assert emissive > 10 and transmissive > 10 and alpha > 10


def test_gltf_material_overrides(product, tmp_path):
    """rtxpt_b200_load_gltf_ex: RTXPT material files replace glTF materials by name, scene-specialised folder before the shared one,
    <model>.<name> before <name>; ExcludeFromNEE / alpha test / SkipRender reach the sub-instance and geometry tables."""
    import gltf_export
    from test_gltf_loader import _textured_builder
    from rtxpt_b200 import structs as S
    b = _textured_builder()
    path = gltf_export.export(b, str(tmp_path / "city.gltf"))
    shared = tmp_path / "Materials"; scene_dir = shared / "demo"; scene_dir.mkdir(parents=True)
    base = product.GltfScene(path)
    over0 = {"BaseOrDiffuseColor": [0.1, 0.2, 0.3], "Roughness": 0.77, "Metalness": 0.5, "ExcludeFromNEE": True, "EnableNormalTexture": False,
             "BaseTexture": {"path": "x\\\\a.dds", "sRGB": True}, "NormalTexture": {"path": "x\\\\n.dds"}}
    (shared / "city.mat0.material.json").write_text(json.dumps(over0))
    (shared / "mat1.material.json").write_text(json.dumps({"Roughness": 0.11, "EnableAlphaTesting": False}))           # <name> only, shared folder
    (shared / "city.mat2.material.json").write_text(json.dumps({"Roughness": 0.99}))                                    # loses against the scene-specialised file below
    (scene_dir / "city.mat2.material.json").write_text(json.dumps({"Roughness": 0.33, "EnableTransmission": True, "TransmissionFactor": 0.5, "IoR": 1.2, "SkipRender": True}))
    g = product.GltfScene(path, materials_dir=str(shared), scene_materials_dir=str(scene_dir))
    assert g.overridden_materials == 3 and g.desc.materialCount == base.desc.materialCount
    m0, m1, m2, m3 = (g.desc.materials[i] for i in range(4))
    assert abs(m0.Roughness - 0.77) < 1e-7 and list(m0.BaseOrDiffuseColor) == [np.float32(0.1), np.float32(0.2), np.float32(0.3)]
    assert m0.Flags & S.MATFLAG_UseBaseOrDiffuseTexture and m0.BaseOrDiffuseTextureIndex == base.desc.materials[0].BaseOrDiffuseTextureIndex      # glTF texture kept where the file enables the slot
    assert not (m0.Flags & S.MATFLAG_UseNormalTexture) and m0.NormalTextureIndex == 0xFFFFFFFF                                                  # ... dropped where it disables it
    assert abs(m1.Roughness - 0.11) < 1e-7 and abs(m2.Roughness - 0.33) < 1e-7 and abs(m2.IoR - 1.2) < 1e-7 and abs(m2.TransmissionFactor - 0.5) < 1e-7
    assert bytes(m3) == bytes(base.desc.materials[3])                                                                                            # untouched
    subs = [g.desc.subInstances[i] for i in range(g.desc.subInstanceCount)]; bsubs = [base.desc.subInstances[i] for i in range(base.desc.subInstanceCount)]
    for s, bs in zip(subs, bsubs):
        mi = s.GlobalGeometryIndex_PTMaterialDataIndex & 0xFFFF
        assert bool(s.FlagsAndAlphaInfo & S.SUBINST_FLAG_EXCLUDE_FROM_NEE) == (mi == 0)
        if mi == 1: assert not (s.FlagsAndAlphaInfo & S.SUBINST_FLAG_ALPHA_TESTED) and (bs.FlagsAndAlphaInfo & S.SUBINST_FLAG_ALPHA_TESTED)   # the file switched the cutout off
    skipped = [g.desc.geometries[i] for i in range(g.desc.geometryCount) if g.desc.geometries[i].materialIndex == 2]
    assert skipped and all(x.numIndices == 0 for x in skipped) and g.triangle_count < base.triangle_count
    g.close(); base.close()
