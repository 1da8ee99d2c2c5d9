"""Writes tests/golden/final_assets_pack.npz and final_assets_tables.json from the reference's own asset directory.

    python tests/golden/make_final_pack.py <the reference checkout's assets/ directory>

The reference's assets are not part of this repository, so config 4 (BASELINE.json: "assets/Final triangle-mesh scene")
is rebuilt from this pack: the tables `parse_obj` / `parse_mtl` produce for the 13 OBJ files the reference ships
(src/main.rs:208-223 names 15; 初音未来.obj and 卒.obj are listed in .MISSING_LARGE_BLOBS), and the decoded RGBA8
texels of the images their MTL files name.  Geometry and materials are stored verbatim (binary64); images are
box-reduced to <= 512 texels on the longer side to keep the fixture small - texture resolution does not change
which code runs (the reference samples them nearest-texel, texture.rs:111-119).
final_assets_tables.json holds the digests of the scene tables obj_scene() builds from the asset directory itself,
which test_final_scene.py::test_pack_equals_reference_files compares with the scene built from the pack.
"""
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
# order of obj_scene(), src/main.rs:208-223 (+ the fog mesh, :224)
OBJ_FILES = ["初音未来.obj", "玻璃球.obj", "外框.obj", "声匣.obj", "镜子门.obj", "镜子.obj", "环.obj", "传送门框.obj", "水下.obj", "水面.obj",
             "文字.obj", "mc.obj", "伞.obj", "卒.obj", "雾.obj"]


def _module(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


if __name__ == "__main__":
    assets = sys.argv[1]
    pkg = os.path.join(ROOT, "raytracer-2025_b200")
    objload = _module("objload", os.path.join(pkg, "objload.py"))
    out = os.path.join(ROOT, "tests", "golden", "final_assets_pack.npz")
    meta = objload.write_pack(out, assets, [("Final", f) for f in OBJ_FILES], max_image_side=512)
    print("objs:", len(meta["objs"]), "mtls:", len(meta["mtls"]), "images:", len(meta["images"]), "bytes:", os.path.getsize(out))
    for k in OBJ_FILES:
        if "Final/" + k not in meta["objs"]:
            print("  missing:", k)
    rt = _module("rt2025", os.path.join(pkg, "rt2025.py"))
    hs, _ = _module("scenes", os.path.join(pkg, "scenes.py")).obj_scene(rt, assets, width=96, spp=4, depth=12)
    digests = _module("scenes_util", os.path.join(ROOT, "tests", "scenes_util.py")).table_digests(hs)
    with open(os.path.join(ROOT, "tests", "golden", "final_assets_tables.json"), "w") as f:
        json.dump(digests, f, indent=1)
        f.write("\n")
    sys.exit(0)
