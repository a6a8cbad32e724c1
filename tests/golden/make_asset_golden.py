"""Generates tests/golden/reference_assets.json.gz from a checkout of the reference (RTXPT at commit f08d1c7): the data files of its Assets tree that
tests/test_material_json.py and tests/test_scene_json.py read, so that those tests run without the reference.
  materials     every Assets/Materials/*.material.json and Assets/Materials/*/*.material.json, as text
  scenes        every Assets/*.scene.json, as text
  models        the model files those scenes name that exist in the checkout (git-LFS pointer stubs there), as text
  scene_errors  what rtxpt_b200_load_scene_json answers for each scene file, with the Assets directory written as {assets}
Needs the product library (rtxpt_b200.lib.build()):
    python tests/golden/make_asset_golden.py <reference checkout>"""
import glob
import gzip
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def read(path):
    with open(path, encoding="utf-8") as f:
        return f.read()


def main(ref):
    from rtxpt_b200 import lib
    assets = os.path.join(os.path.abspath(ref), "Assets")
    rel = lambda p: os.path.relpath(p, assets).replace(os.sep, "/")
    mats = sorted(glob.glob(os.path.join(assets, "Materials", "*.material.json")) + glob.glob(os.path.join(assets, "Materials", "*", "*.material.json")))
    scenes = sorted(glob.glob(os.path.join(assets, "*.scene.json")))
    data = {"materials": {rel(p): read(p) for p in mats}, "scenes": {rel(p): read(p) for p in scenes}, "models": {}, "scene_errors": {},
            "_source": "Assets/ of the reference at commit f08d1c7 (tests/golden/make_asset_golden.py)"}
    for p in scenes:
        try:
            names = json.loads(read(p)).get("models", [])
        except ValueError:
            names = []
        for m in names:
            mp = os.path.join(assets, m.replace("\\", "/"))
            if os.path.isfile(mp):
                data["models"][rel(mp)] = read(mp)
        try:
            lib.GltfScene(p).close()
            raise SystemExit("%s loaded; expected its model stubs to be refused" % p)
        except lib.RtxptError as e:
            data["scene_errors"][rel(p)] = str(e).replace(assets, "{assets}")
    out = os.path.join(ROOT, "tests", "golden", "reference_assets.json.gz")
    with gzip.GzipFile(out, "wb", mtime=0) as f:
        f.write(json.dumps(data, indent=0, sort_keys=True).encode())
    print({k: len(v) for k, v in data.items() if isinstance(v, dict)}, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
