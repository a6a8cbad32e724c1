"""CPU: the oracle's integer / packing primitives against the reference's own known answers.
  - tests/golden/rng_golden.json: produced from the UNMODIFIED NoiseAndSequences.hlsli C++ half (tests/golden/make_rng_golden.py)
  - fp16 known answers of External/Donut/tests/src/engine/test_float.cpp:74-90 (round-to-nearest-even f32->f16)
  - where build() compiled oracle/_ref/ from the reference sources, the golden file is regenerated and must be identical (pins the fixture itself)"""
import json
import os
import subprocess
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def golden():
    with open(os.path.join(HERE, "golden", "rng_golden.json")) as f:
        return json.load(f)


def test_hash32_against_reference_header(oracle):
    L = oracle.lib(); g = golden()
    for x, h in g["hash32"]:
        assert L.oracle_hash32(x) == h
    for s, v, h in g["hash32_combine"]:
        assert L.oracle_hash32_combine(s, v) == h
    for h, f in g["hash32_to_float"]:
        assert np.float32(L.oracle_hash32_to_float(h)) == np.float32(f)
        assert 0.0 <= f < 1.0


def test_sobol_against_reference_header(oracle):
    L = oracle.lib()
    for index, dim, v in golden()["sobol"]:
        assert L.oracle_sobol(index, dim) == v


def _ref_binary(name):
    """oracle/_ref/<name>, compiled by build() (make -C oracle ref) where the reference sources are present; the test skips where it was never built."""
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "ref"], check=True)
    exe = os.path.join(ROOT, "oracle", "_ref", name)
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/%s not built (build() compiles it only where the reference sources are present)" % name)
    return exe


def test_golden_file_matches_reference_tree():
    out = subprocess.run([_ref_binary("ref_kat")], check=True, capture_output=True, text=True).stdout
    fresh = json.loads(out); g = golden()
    for k in ("hash32", "hash32_combine", "sobol"):
        assert fresh[k] == g[k]


def test_fp16_known_answers_from_donut_test_float(oracle):
    L = oracle.lib()
    inv1024 = np.float32(1.0 / 1024.0); smallest_normal = np.float32(2.0 ** -14)
    cases = [(0.0, 0), (smallest_normal * inv1024 * np.float32(0.5), 0), (smallest_normal * inv1024, 1), (smallest_normal * inv1024 * np.float32(1023.0), 0x03ff),
             (np.float32(1.0) / np.float32(3.0), 0x3555), (np.float32(0.5) * (np.float32(1.0) + np.float32(1023.0) / np.float32(1024.0)), 0x3bff), (1.0, 0x3c00),
             (np.float32(1.0) + inv1024, 0x3c01), (65504.0, 0x7bff), (np.inf, 0x7c00), (-np.inf, 0xfc00), (65519.0, 0x7bff), (65520.0, 0x7c00), (1000000.0, 0x7c00)]
    for v, bits in cases:
        assert L.oracle_f32tof16(float(v)) == bits, (v, bits)
    assert (L.oracle_f32tof16(float("nan")) & 0x7c00) == 0x7c00 and (L.oracle_f32tof16(float("nan")) & 0x3ff) != 0


def test_fp16_matches_ieee_rne_exhaustively_sampled(oracle):
    L = oracle.lib()
    rng = np.random.default_rng(0)
    bits = np.concatenate([rng.integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32),
                           (np.arange(0, 65536, dtype=np.uint32) << 13) + 0x38000000])     # around the f16 normal range, incl. exact ties
    vals = bits.view(np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        ref = vals.astype(np.float16).view(np.uint16)
    for v, r in zip(vals[:60000], ref[:60000]):
        if np.isnan(v):
            continue
        assert L.oracle_f32tof16(float(v)) == int(r)
    # all 65536 halves round-trip
    for h in range(0, 65536, 7):
        f = L.oracle_f16tof32(h)
        if np.isnan(f):
            continue
        assert L.oracle_f32tof16(f) == h


def test_snorm8_roundtrip(oracle):
    L = oracle.lib()
    for q in range(-127, 128):
        assert L.oracle_pack_snorm8(L.oracle_unpack_snorm8(q & 0xff)) == (q & 0xff)
    assert L.oracle_unpack_snorm8(0x80) == -1.0     # -128 clamps


def test_sample_sequences_are_in_unit_interval_and_deterministic(oracle):
    L = oracle.lib()
    rng = np.random.default_rng(1)
    tuples = np.stack([rng.integers(0, 1920, 4096), rng.integers(0, 1080, 4096), rng.integers(0, 8, 4096), rng.integers(0, 5000, 4096)], 1).astype(np.uint32)
    out = np.zeros((4096, 8), np.uint32); out2 = np.zeros_like(out)
    L.oracle_rng(tuples.ctypes.data, 4096, out.ctypes.data); L.oracle_rng(tuples.ctypes.data, 4096, out2.ctypes.data)
    assert np.array_equal(out, out2)
    ld = out[:, 4:].view(np.float32)
    assert (ld >= 0).all() and (ld < 1).all()
    # uniform stream: chained Hash32 of the seeded state (StatelessSampleGenerators.hlsli:187-232)
    x, y, v, s = [int(t) for t in tuples[0]]
    base = L.oracle_hash32_combine(L.oracle_hash32((v + 0x035F9F29) & 0xFFFFFFFF), (x << 16) | y)
    h = L.oracle_hash32_combine(L.oracle_hash32_combine(base, 0), s)
    for k in range(4):
        h = L.oracle_hash32(h); assert out[0, k] == h
    # low-discrepancy draws are stratified: first dimension over sample indices 0..255 of one pixel covers every 1/256 stratum exactly once
    t = np.array([[10, 20, 1, i] for i in range(256)], np.uint32); o = np.zeros((256, 8), np.uint32)
    L.oracle_rng(t.ctypes.data, 256, o.ctypes.data)
    strata = np.floor(o[:, 4].view(np.float32) * 256).astype(int)
    assert len(set(strata.tolist())) == 256


# ---- floating-point material model: pinned to the reference's own HLSL headers compiled in place (tests/golden/make_bsdf_golden.py) --------------------------------------
def bsdf_golden():
    return np.load(os.path.join(HERE, "golden", "bsdf_golden.npz"))


def _same(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


def test_standard_bsdf_equals_the_reference_headers_bit_for_bit(oracle):
    """eval / evalPdf / sample / getLobes / evalDeltaLobes / estimateSpecDiffBSDF of oracle/pt_bsdf.h against StandardBSDF.hlsli + BxDF.hlsli themselves: every one of the 40 outputs
    of every record identical.  (g++ on both sides, IEEE binary32, no contraction, the same libm: what differs between the two builds is only who wrote the formulas.)"""
    import ctypes as C
    g = bsdf_golden(); L = oracle.lib()
    L.oracle_bsdf_ex.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_bsdf_ex.restype = None
    rec = np.ascontiguousarray(g["bsdf_in"], np.float32); out = np.zeros((len(rec), 40), np.float32)
    L.oracle_bsdf_ex(rec.ctypes.data, len(rec), out.ctypes.data)
    ref = g["bsdf_out"]
    bad = ~_same(out, ref)
    assert not bad.any(), (int(bad.sum()), np.unique(np.where(bad)[1]), np.abs(out - ref)[bad].max())
    # the fixture exercises what it claims to: all four lobe kinds sampled, delta and rough, valid and rejected samples, both delta lobes
    lobes = ref[ref[:, 5] > 0, 13].astype(int)
    assert all((lobes & m).any() for m in (0x01, 0x02, 0x04, 0x10, 0x20, 0x40)) and (ref[:, 5] == 0).sum() > 20
    assert (ref[:, 19] > 0).sum() > 100 and (ref[:, 27] > 0).sum() > 100 and (ref[:, 34:40] > 0).any()


def test_material_building_blocks_equal_the_reference_headers_bit_for_bit(oracle):
    """Fresnel.hlsli, Microfacet.hlsli, MathHelpers.hlsli functions the live path calls; slots the oracle does not restate (unused by the path) come back NaN and are skipped."""
    import ctypes as C
    g = bsdf_golden(); L = oracle.lib()
    L.oracle_bsdf_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_bsdf_funcs.restype = None
    u = np.ascontiguousarray(g["funcs_in"], np.float32); out = np.zeros((len(u), 40), np.float32)
    L.oracle_bsdf_funcs(u.ctypes.data, len(u), out.ctypes.data)
    ref = g["funcs_out"]
    restated = ~np.isnan(out).all(0)
    assert restated.sum() >= 34
    bad = ~_same(out[:, restated], ref[:, restated])
    assert not bad.any(), (int(bad.sum()), np.where(restated)[0][np.unique(np.where(bad)[1])])


def test_bsdf_golden_file_matches_reference_tree():
    _ref_binary("ref_kat_bsdf")
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_bsdf_golden", os.path.join(HERE, "golden", "make_bsdf_golden.py")); m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    rec, out, u, fout = m.generate(); g = bsdf_golden()
    assert np.array_equal(rec, g["bsdf_in"]) and _same(out, g["bsdf_out"]).all() and np.array_equal(u, g["funcs_in"]) and _same(fout, g["funcs_out"]).all()


def test_utils_functions_match_reference_header_golden(oracle):
    """Utils/Utils.hlsli compiled in place (tests/golden/make_utils_golden.py): the balance heuristic of every MIS weight on the path, the octahedral normal encodings of the
    stable planes and of the light records (32- and 30-bit packings), FastSqrt / FastACos - the oracle's restatements reproduce the reference's outputs bit for bit (NaN where
    the reference yields NaN)."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "utils_golden.npz"))
    u, ref = np.ascontiguousarray(g["utils_in"]), g["utils_out"]
    L = oracle.lib(); L.oracle_utils_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_utils_funcs.restype = None
    out = np.empty_like(ref); L.oracle_utils_funcs(u.ctypes.data, len(u), out.ctypes.data)
    restated = [3, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20]      # EvalMIS(Balance); Encode_Oct; Decode_Oct; NDirToOctUnorm32; OctToNDirUnorm32; ..Unorm30 both ways; FastSqrt; FastACos
    for k in restated:
        same = (out[:, k].view(np.uint32) == ref[:, k].view(np.uint32)) | (np.isnan(out[:, k]) & np.isnan(ref[:, k]))
        assert same.all(), (k, int((~same).sum()))
    assert np.isnan(out[:, [0, 1, 2, 4, 5, 21, 22, 23]]).all()                  # not restated (unused by the live path): LuminanceClamp, power / three-way MIS, WeightedAverage, ...


def test_path_tracer_helpers_match_reference_header_golden(oracle):
    """PathTracerHelpers.hlsli compiled in place (tests/golden/make_helpers_golden.py): the self-intersection offset of every ray origin (ComputeRayOrigin), the grazing-angle
    fade-out of NEE, the ray-cone growth by scatter pdf, the firefly-filter K update and both firefly filters, the balance heuristic - bit for bit.  (The firefly filter's lpfloat
    arithmetic rounds to binary16 after EVERY operation; the restatement had rounded once per expression until this vector set caught it: 44 % of the filtered values were off by
    1-2 fp16 steps.)"""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "helpers_golden.npz"))
    u, ref = np.ascontiguousarray(g["helpers_in"]), g["helpers_out"]
    L = oracle.lib(); L.oracle_helper_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_helper_funcs.restype = None
    out = np.empty_like(ref); L.oracle_helper_funcs(u.ctypes.data, len(u), out.ctypes.data)
    for k in (0, 1, 2, 3, 7, 8, 9, 10, 11, 12, 13, 14, 15):                    # 14, 15: two fixed linear combinations of MatrixRotateFromTo's nine entries
        same = (out[:, k].view(np.uint32) == ref[:, k].view(np.uint32)) | (np.isnan(out[:, k]) & np.isnan(ref[:, k]))
        assert same.all(), (k, int((~same).sum()))
    assert (ref[:, 9:12] != np.float32(u[:, 0:3] * 8).astype(np.float16).astype(np.float32)).any(1).mean() > 0.2       # the filter did clamp a good share of the records


def test_triangle_light_matches_reference_header_golden(oracle):
    """Lighting/PolymorphicLight.hlsli compiled in place (tests/golden/make_lights_golden.py): TriangleLight::Store - the 32-byte record LightsBaker writes for every emissive
    triangle (PackColor's log radiance + R8G8B8 colour, centre, half-packed edges) -, Create, CalcSample (uniform triangle sample + ComputeRayOrigin + area -> solid-angle pdf),
    CalcSolidAnglePdfForMIS and GetPower: the oracle reproduces all of it bit for bit.  This includes a quirk of the reference: Store holds the packed edge words in a `float3`
    before writing them (uint -> float -> uint), so each word keeps only 24 significant bits and edge1 loses its low mantissa bits; the restatement now does the same."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "lights_golden.npz"))
    u, ref = np.ascontiguousarray(g["lights_in"]), g["lights_out"]
    L = oracle.lib(); L.oracle_light_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_light_funcs.restype = None
    out = np.empty_like(ref); L.oracle_light_funcs(u.ctypes.data, len(u), out.ctypes.data)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))
    assert same.all(), same.mean(0)
    # the quirk is real in these vectors: the stored edge1 differs from the half-rounded input on most records
    e1 = u[:, 3:6].astype(np.float16).astype(np.float32)
    rel = np.abs(ref[:, 20:23] - e1) / (np.abs(e1) + 1e-6)
    assert (ref[:, 20:23] != e1).any(1).mean() > 0.9 and 0.005 < np.median(rel) < 0.03 and np.percentile(rel, 99) < 0.15           # measured: median 1.8 %, 99th percentile 10 % of the component


def test_sphere_light_matches_reference_header_golden(oracle):
    """The analytic sphere / spot light of Lighting/PolymorphicLight.hlsli + LightShaping.hlsli compiled in place: the record (PackColor, half radius, oct-packed axis, half cone
    cosines), SphereLight::Create, the dispatcher's CalcSample (cone sampling of the visible cap x evaluateLightShaping), CalcSolidAnglePdfForMIS and GetPower (the weight the
    proxy table is built from) - bit for bit, including a viewer inside the sphere.  (GetPower's product is associated as getSurfaceArea() = 4 pi sq(r) first; the restatement's
    4 pi r r was 1 ulp off on a fifth of the records until these vectors caught it.)"""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "sphere_lights_golden.npz"))
    u, ref = np.ascontiguousarray(g["spheres_in"]), g["spheres_out"]
    L = oracle.lib(); L.oracle_sphere_light_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_sphere_light_funcs.restype = None
    out = np.empty_like(ref); L.oracle_sphere_light_funcs(u.ctypes.data, len(u), out.ctypes.data)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))
    assert same.all(), same.mean(0)
    assert (ref[:, 21] > 0).mean() > 0.9 and (u[:, 7] > 0.5).mean() > 0.3 and ((ref[:, 18:21] == 0).all(1) & (u[:, 7] > 0.5)).mean() > 0.05        # spots exist and some viewers sit outside their cone


def test_tone_mapping_operators_match_reference_shader_golden(oracle):
    """Rtxpt/ToneMapper/ToneMapping.ps.hlsli compiled in place (tests/golden/make_tonemap_golden.py): Linear, Reinhard, ReinhardModified, HejiHableAlu, HableUc2 and Aces through
    toneMap(), and calcLuminance - the oracle's operators (pt_tonemap.h, which the CUDA tone mapper reproduces byte for byte in tests/test_gpu_tonemap.py) are the reference's
    bit for bit, NaN for NaN on black input."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "tonemap_golden.npz"))
    u, ref = np.ascontiguousarray(g["tonemap_in"]), g["tonemap_out"]
    L = oracle.lib(); L.oracle_tonemap_ops.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_tonemap_ops.restype = None
    out = np.empty_like(ref); L.oracle_tonemap_ops(u.ctypes.data, len(u), out.ctypes.data)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))
    assert same.all(), same.mean(0)
    assert all((u[:, 3] == op).sum() > 300 for op in range(6))


def test_ray_cone_texture_lod_matches_reference_header_golden(oracle):
    """Rendering/Materials/TexLODHelpers.hlsli compiled in place (tests/golden/make_texlod_golden.py): the fp16-packed ray cone, its propagation over a segment, the per-triangle
    LOD constant (texture-space over world-space area through the instance matrix) and computeLOD with and without the slope term - every material texture fetch of the path
    takes its MIP level from these; bit for bit, including the clamped logarithm of degenerate texture triangles."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "texlod_golden.npz"))
    u, ref = np.ascontiguousarray(g["texlod_in"]), g["texlod_out"]
    L = oracle.lib(); L.oracle_texlod_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_texlod_funcs.restype = None
    out = np.empty_like(ref); L.oracle_texlod_funcs(u.ctypes.data, len(u), out.ctypes.data)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))
    assert same.all(), same.mean(0)
    assert (ref[:40, 0] < -60).all() and np.isfinite(ref).all()


def test_interior_list_matches_reference_header_golden(oracle):
    """Rendering/Materials/InteriorList.hlsli compiled in place (tests/golden/make_interior_golden.py): the two-slot stack of nested dielectrics through 12 surface crossings per
    record - well-formed enter / leave sequences as closed meshes produce them, and random ones (a full stack, leaving a medium that was never entered, priority 0) - slots,
    top / next material, top priority and the true-intersection test agree after every crossing."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "interior_golden.npz"))
    u, ref = np.ascontiguousarray(g["interior_in"]), g["interior_out"]
    L = oracle.lib(); L.oracle_interior_list.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_interior_list.restype = None
    out = np.empty_like(ref); L.oracle_interior_list(u.ctypes.data, len(u), out.ctypes.data)
    assert (out.view(np.uint32) == ref.view(np.uint32)).all()
    r = ref.reshape(len(u), 12, 6)
    assert (r[:2000, -1, 0].view(np.uint32) == 0).mean() > 0.5 and (r[..., 5] == 0).mean() > 0.05 and (r[..., 4] >= 0).mean() > 0.2        # stacks unwind; false intersections and two-deep stacks occur


def test_light_sampler_matches_reference_header_golden(oracle):
    """Lighting/LightSampler.hlsli, LightingTypes.hlsli's LightFeedbackReservoir and LightingAlgorithms.hlsli's LocalLightBinarySearch compiled in place with CPU stand-ins for
    the resource views (tests/golden/make_sampler_golden.py): 1200 scenarios of 16 lights, <= 64 global proxies, 2 x 2 tiles and 8 queries each.  SampleGlobal / SampleLocal,
    both selection pdfs, the candidate split, the MIS weights on either side, the feedback reservoir after InsertFeedbackFromNEE and the coherence heuristic agree bit for bit -
    including the binary search's behaviour for a light below every key of the tile (step 8 reads the previous tile's last entry; tile 0 reads out of range = "light 0, 1")."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "sampler_golden.npz"))
    u, ref = np.ascontiguousarray(g["sampler_in"]), g["sampler_out"]
    L = oracle.lib(); L.oracle_sampler_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_sampler_funcs.restype = None
    out = np.empty_like(ref); L.oracle_sampler_funcs(u.ctypes.data, len(u), out.ctypes.data)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))          # 0 / 0 MIS weights (delta lobe against a light without proxies) are NaN on both sides
    assert same.all()
    r = ref.reshape(len(u), 8, 16); q = u[:, 600:].reshape(len(u), 8, 10)
    quirk = r[1100:, [5, 7], 5]                                                                      # the generator's constructed cases: tile 0 / light 0, tile 1 / tile 0's last key
    assert (quirk[:, 0] == np.float32(1 / 128)).all() and (quirk[:, 1] > 0).all()
    assert (r[:1100, :, 5] > 0).mean() > 0.3 and (r[:1100, :, 5] == 0).mean() > 0.2 and (r[..., 6] > 0).mean() > 0.2 and (r[..., 13] > 0).mean() > 0.95
    assert ((r[..., 14].view(np.uint32) & 0x7FFFFFFF) == q[..., 3].astype(np.uint32)).mean() > 0.5      # most inserts win their (mostly empty) reservoir


def test_handle_hit_matches_reference_path_tracer_golden(oracle):
    """PathTracer::HandleHit of the UNMODIFIED PathTracer.hlsli - with PathTracerNEE.hlsli (candidate loop, weighted reservoir, shadow ray, both MIS weights, firefly filter, fp16
    accumulation, NEE-AT feedback), PathTracerNestedDielectrics.hlsli (false-hit rejection, outside IoR), GenerateScatterRay (BSDF sample, ray cone, bounce counters, firefly K),
    HandleRussianRoulette, the Sobol / hash sample generators and the 80-byte path payload - compiled in place behind a stub bridge (oracle/ref_bridge_stub.h,
    tests/golden/make_hit_golden.py) three times, as the three shaders RTXPT compiles it into:
      reference mode;
      the BUILD pass (PathTracerStablePlanes.hlsli's StablePlanesHandleHit: delta-lobe enumeration, plane allocation, SplitDeltaPath with the accumulated image transform,
        StablePlanes.hlsli's StoreStablePlane / StoreExplorationStart packing, dominant plane, stable radiance);
      the FILL pass (StablePlanesOnScatter, CommitDenoiserRadiance, the specular hit distance, attenuated noisy radiance).
    1200 path vertices each, a quarter of them rays that leave the scene (HandleMiss: environment lookup, MIS against the environment-quad light, StablePlanesHandleMiss), lights of all
    three kinds in the NEE-AT tables; plus the per-pixel driver's own steps (PathTracer::EmptyPathInitialize, PathTracerSample.hlsl's FirstHitFromVBuffer - the FILL pass restarting from
    plane 0 as the BUILD records stored it - and postProcessHit - the BUILD pass picking up the next enqueued branch): the outgoing payload, the shadow ray, the feedback reservoir, the pixel's three stable planes (all 80 bytes), its header and stable radiance and the hit
    distance the oracle's HandleHitSurface produces are bit-identical."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "hit_golden.npz"))
    L = oracle.lib(); L.oracle_hit_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]; L.oracle_hit_funcs.restype = None
    for key, mode in (("hit", 0), ("build", 1), ("fill", 2)):
        u, ref = np.ascontiguousarray(g[key + "_in"]), g[key + "_out"]
        out = np.empty_like(ref); L.oracle_hit_funcs(u.ctypes.data, len(u), out.ctypes.data, mode)
        same = out.view(np.uint32) == ref.view(np.uint32); same[:, 35:37] = True            # 35, 36: how often the bridge's ExportSpecHitTStart / Stop were called (not mirrored)
        if mode == 1: same[:, 30] = True; same[:, 32:35] = True; same[:, 117:120] = True    # what Bridge::ExportSurface / ExportNonSurface were handed (the stub records it; the planes hold the same values packed)
        assert same.all(), (key, np.argwhere(~same)[:8])
        R, U = ref.view(np.uint32), u.view(np.uint32); p, pin = R[:, :20], U[:, :20]
        hitv = u[:, 27] == 0; missv = u[:, 27] == 1
        assert 200 < missv.sum() < 400 and ((R[missv, 19] >> 10) & 1).max() == 0                # a miss ends the path
        if mode != 1: assert (R[missv, 10:12] != U[missv, 10:12]).any(1).mean() > 0.3            # ... and adds the environment's radiance
        else: assert (R[missv, 47:50] != U[missv, 920:923]).any(1).all()                         # ... BUILD stores the sky as a plane
        assert (u[:, 27] == 2).sum() == 60                                                       # EmptyPathInitialize
        if mode == 2: m3 = u[:, 27] == 3; assert m3.sum() == 240 and 10 < np.isinf(u[m3, 967]).sum() < 200 and (ref[m3, 120] > 0).sum() > 40       # FirstHitFromVBuffer: sky planes (inline miss) and surfaces (bracketed ray)
        if mode == 1: m4 = u[:, 27] == 4; assert m4.sum() == 200 and 0.3 < (R[m4, 47:50] != U[m4, 920:923]).any(1).mean() < 0.95                    # postProcessHit: an ended path picks up the next enqueued branch, a live one does not
        if mode != 1:   # one and two shadow rays, occluded and visible, radiance added, paths ending and going on, feedback written
            assert np.bincount(ref[:, 20].astype(int), minlength=3)[1:3].min() > 80 and 0.2 < ref[:, 28].mean() < 0.6 and (ref[:, 39] > 0).mean() > 0.15
            assert (p[hitv, 10:12] != pin[hitv, 10:12]).any(1).mean() > 0.3 and 0.05 < 1 - ((p[hitv, 19] >> 10) & 1).mean() < 0.5 and (p[hitv, 8:10] != pin[hitv, 8:10]).any(1).mean() > 0.8
        if mode == 0: assert (ref[hitv, 29] == 0).sum() > 8                                 # rejected false hits export nothing
        if mode == 2:   # landing on a stable plane commits the path's radiance into it; specular hit distances start and stop
            assert (R[:, 41:47] != U[:, 924:930]).any(1).sum() > 30 and (ref[:, 37] != u[:, 930]).sum() > 120 and ref[:, 35].sum() > 50
        if mode == 1:   # planes enqueued for later exploration, paths that keep walking the delta tree (new branch id, turned image transform), base planes stored, stable emission
            hin, hout = U[:, 920:924], R[:, 47:51]
            assert ((hout[:, :3] == 0xFFFFFFFE) & (hin[:, :3] != 0xFFFFFFFE)).any(1).mean() > 0.1 and (R[:, 15] != U[:, 15]).mean() > 0.05 and (R[:, 10:12] != U[:, 10:12]).any(1).mean() > 0.03
            assert 1 - ((R[:, 19] >> 10) & 1).mean() > 0.7 and (ref[:, 52:55] != u[:, 946:949]).any(1).mean() > 0.15 and 0.3 < ref[:, 29].mean() < 0.8


def test_environment_quad_light_matches_reference_header_golden(oracle):
    """Lighting/PolymorphicLight.hlsli's EnvironmentQuadLight compiled in place (tests/golden/make_hit_golden.py, mode "envquads"): Store (the record of a quad-tree node over the
    equal-area octahedral environment map), Create, the sample NEE draws from a node through the environment's rotation, its solid-angle pdf and power - bit for bit."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "envquad_lights_golden.npz"))
    u, ref = np.ascontiguousarray(g["envquads_in"]), g["envquads_out"]
    L = oracle.lib(); L.oracle_envquad_light_funcs.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_envquad_light_funcs.restype = None
    out = np.empty_like(ref); L.oracle_envquad_light_funcs(u.ctypes.data, len(u), out.ctypes.data)
    assert (out.view(np.uint32) == ref.view(np.uint32)).all()
    assert np.allclose(np.linalg.norm(ref[:, 15:18], axis=1), 1, atol=1e-4) and (ref[:, 21] == (u[:, 2] ** 2 / np.float32(4 * np.pi)).astype(np.float32)).mean() > 0.9


def test_neeat_feedback_passes_match_reference_lights_baker_golden(oracle):
    """NEE-AT's frame-end passes of the UNMODIFIED Rtxpt/Lighting/LightsBaker.hlsl compiled in place (tests/golden/make_baker_golden.py, oracle/_ref/ref_kat_baker; the passes of
    LightsBaker::UpdateEnd but PreFilter, whose in-place update races across thread groups): ProcessFeedbackHistoryP0 (remap to this frame's light list, per-light usage counters, world-space candidates stripped),
    P1a (the half-resolution blend through depth / motion reprojection), P1b (full-resolution reservoirs: reprojected + blended, holes filled from last frame's tile or the global
    table), P2 / FillTile (the 8 x 8 window + 64 top-up picks per tile), P3 (the bitonic sort in group-shared memory and the duplicate counts - run on 64 real threads with a barrier behind
    GroupMemoryBarrierWithGroupSync) and ClearFeedbackHistory (the faded seed of next frame's reservoirs, history depth).  200 frames on a 16 x 16
    image, 16 lights: every reservoir, counter, tile entry and depth the oracle's passes produce is bit-identical."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "baker_golden.npz"))
    u, ref = np.ascontiguousarray(g["baker_in"]), g["baker_out"]
    L = oracle.lib(); L.oracle_baker_feedback.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_baker_feedback.restype = None
    out = np.zeros_like(ref); L.oracle_baker_feedback(u.ctypes.data, len(u), out.ctypes.data)
    same = out.view(np.uint32) == ref.view(np.uint32)
    assert same.all(), np.argwhere(~same)[:8]
    R, U = ref.view(np.uint32), u.view(np.uint32)
    # P0 strips and remaps, the reprojection both finds and loses its pixel, holes get filled, the seed keeps part of the history
    assert 0.3 < ((R[:, 256:512] == 0xFFFFFFFF) & (U[:, 368:624] != 0xFFFFFFFF)).mean() < 0.7 and 0.3 < (ref[:, 657:913] > 0).mean() < 0.7 and (R[:, 913:1169] != 0xFFFFFFFF).all()
    assert (ref[:, 2321:2577] > 0).mean() > 0.4 and (ref[:, 512:529].sum(1) == 256).all()
    lists = R[:, 3089:4241].reshape(-1, 128); assert (np.diff((lists >> 9).astype(np.int64), axis=1) >= 0).all() and ((lists & 0x1FF) > 0).mean() > 0.9       # sorted, duplicates counted


def test_neeat_proxy_counts_match_reference_lights_baker_golden(oracle):
    """ComputeProxyCounts of the UNMODIFIED LightsBaker.hlsl (UpdateBegin: every light's share of the global sampling proxies from its weight blended with last frame's usage
    counters; one thread per light, a group barrier, thread 0 sums - run on real threads): 1000 light lists incl. unused lights, a light 10^4 times brighter than the rest (the
    per-light cap), uniform sampling, no valid feedback at all.  Counters, offsets and the total are bit-identical with the oracle's RebuildGlobalProxies."""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "baker_golden.npz"))
    u, ref = np.ascontiguousarray(g["counts_in"]), g["counts_out"]
    L = oracle.lib(); L.oracle_baker_counts.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]; L.oracle_baker_counts.restype = None
    out = np.zeros_like(ref); L.oracle_baker_counts(u.ctypes.data, len(u), out.ctypes.data)
    assert (out.view(np.uint32) == ref.view(np.uint32)).all()
    assert (ref[:, :16] == 262143).sum() > 100 and (ref[:, 16] == ref[:, 33]).all() and (ref[u[:, 4] == 0, :16].max() <= 60)
