"""Small scene builders shared by the CPU and GPU tests (all through the host mirror)."""
import numpy as np


def _pkg_module(rt, name):
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(name, os.path.join(os.path.dirname(rt.__file__), name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def final_reduced_scene(rt, width=96, spp=4, depth=12):
    """BASELINE.json config 4 on the assets the reference ships: obj_scene() (src/main.rs:207-382) built from
    tests/golden/final_assets_pack.npz (13 of the 15 OBJ files, their MTL records and images; make_final_pack.py),
    with the generated HDR equirect environment in place of assets/13.hdr."""
    import os
    pack = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "final_assets_pack.npz")
    hs, missing = _pkg_module(rt, "scenes").obj_scene(rt, _pkg_module(rt, "objload").AssetPack(pack), width=width, spp=spp, depth=depth)
    assert missing == ["初音未来.obj", "卒.obj"], missing  # .MISSING_LARGE_BLOBS
    return hs


def table_digests(hs):
    """{table: [record count, SHA-256 of its bytes]} for the flat tables of a host scene that do not depend on image
    resolution (the texel pool does)."""
    import ctypes as C
    import hashlib
    d = hs.desc.contents
    return {field: [n, hashlib.sha256(C.string_at(getattr(d, field), n * size)).hexdigest()]
            for field, n, size in (("objects", d.n_objects, 72), ("children", d.n_children, 4), ("planars", d.n_planars, 144),
                                   ("materials", d.n_materials, 176), ("remaps", d.n_remaps, 200), ("transforms", d.n_transforms, 80),
                                   ("textures", d.n_textures, 80))}


def random_graph_scene(rt, seed, n_prims=60, with_transforms=True, with_media=False, with_lights=True, width=24, spp=4, depth=6):
    """A random object graph mixing every container the reference has."""
    rng = np.random.default_rng(seed)
    b = rt.Builder(seed)
    mats = [
        b.lambertian(b.solid(*rng.uniform(0.2, 0.9, 3))),
        b.lambertian(b.checker(0.7, b.solid(0.9, 0.9, 0.9), b.solid(0.1, 0.3, 0.1))),
        b.metal(rng.uniform(0.5, 1, 3), 0.2),
        b.dielectric(b.solid(1, 1, 1), 1.5),
        b.lambertian(b.noise(1.3)),
        b.empty(),
    ]
    light_mat = b.diffuse_light(b.solid(6, 6, 6))

    def prim():
        k = rng.integers(0, 3)
        m = mats[rng.integers(0, len(mats))]
        c = rng.uniform(-4, 4, 3)
        if k == 0:
            return b.sphere(c, rng.uniform(0.2, 0.9), m)
        u, v = rng.uniform(-1.5, 1.5, 3), rng.uniform(-1.5, 1.5, 3)
        if k == 1:
            return b.quad(c, u, v, m)
        return b.triangle(c, u, v, m)

    prims = [prim() for _ in range(n_prims)]
    third = n_prims // 3
    top = []
    top.append(b.bvh(prims[:third]))
    inner = b.list(prims[third:2 * third])
    if with_transforms:
        q = b.quat_axis_angle(rng.normal(size=3), rng.uniform(0, 360))
        inner = b.transform(inner, offset=rng.uniform(-1, 1, 3), quat=q, scale=[1.7, 1.7, 1.7])
    top.append(inner)
    rest = prims[2 * third:]
    if with_transforms:
        q2 = b.quat_axis_angle([0, 1, 0], 33.0)
        sub = b.transform(b.bvh(rest[: len(rest) // 2]), offset=[0.5, -0.5, 1.0], quat=q2)
        top.append(sub)
        top.extend(rest[len(rest) // 2:])
    else:
        top.extend(rest)
    light_quad = b.quad([-1.5, 5.5, -1.5], [3, 0, 0], [0, 0, 3], light_mat)
    top.append(light_quad)
    if with_media:
        top.append(b.medium(b.sphere([0, 0, 0], 3.0, b.empty()), 0.4, b.solid(0.8, 0.8, 0.9)))
        top.append(b.medium(b.box([-6, -6, -6], [6, 6, 6], b.empty()), 0.02, b.solid(1, 1, 1)))
    world = b.list(top)
    lights = rt.RT_NONE
    if with_lights:
        ls = [b.quad([-1.5, 5.5, -1.5], [3, 0, 0], [0, 0, 3], b.empty()), b.sphere([2.5, 2.0, 0.0], 0.6, b.empty())]
        lights = b.list(ls)
    bg = b.gradient([0.05, 0.05, 0.05], [0.1, 0.15, 0.3])
    hs = b.finish(world, lights, width=width, spp=spp, max_depth=depth, vfov=55.0, look_from=(0, 1, 11), look_at=(0, 0, 0),
                  background=bg)
    hs._builder = b
    return hs


def random_rays(rng, n, extent=6.0, time=True):
    o = rng.uniform(-extent, extent, (n, 3))
    d = rng.normal(size=(n, 3))
    t = rng.uniform(0, 1, n) if time else None
    return o, d, t


def scene_rays(rt, orc, hs, n, seed):
    """Half camera rays, half incoherent rays through the scene volume."""
    rng = np.random.default_rng(seed)
    cam = hs.camera
    px = np.stack([rng.integers(0, cam.image_width, n // 2), rng.integers(0, cam.image_height, n // 2)], axis=1)
    prim = orc.camera_rays(cam, 5, px, 0)
    return prim


def compare_hits(rt, got, want, rel=0.0):
    """IDs bit-exact; t bit-exact by default (the north star allows 1e-5 relative): every primitive,
    transformed or not, is intersected with the reference's own binary64 arithmetic."""
    assert np.array_equal(got["prim_id"], want["prim_id"]), \
        f"{int((got['prim_id'] != want['prim_id']).sum())} primitive id mismatches"
    assert np.array_equal(got["inst_id"], want["inst_id"])
    hit = want["prim_id"] != rt.RT_NONE
    if hit.any():
        err = np.abs(got["t"][hit] - want["t"][hit]) / np.abs(want["t"][hit])
        assert err.max() <= rel, f"t relative error {err.max():.3e}"
        # u, v go through acos/atan2 for spheres: libm last-bit differences only
        assert np.abs(got["u"][hit] - want["u"][hit]).max() < 1e-6
        assert np.abs(got["v"][hit] - want["v"][hit]).max() < 1e-6
    assert np.all(np.isinf(got["t"][~hit]))


def materials_scene(rt):
    """Every material / texture / light kind of configs 1-3 plus Mix, Transparent, Portal, checker, image (nearest + bilinear),
    triangle and transformed lights, a defocus camera."""
    rng = np.random.default_rng(7)
    b = rt.Builder(3)
    tex_img = b.image(rng.uniform(0, 1, (16, 8, 4)).astype(np.float32))
    tex_raw = b.image(rng.uniform(0, 1, (5, 7, 4)).astype(np.float32), raw=True)
    white = b.lambertian(b.solid(0.8, 0.8, 0.8))
    mats = [
        b.lambertian(tex_img), b.lambertian(tex_raw), b.lambertian(b.checker(0.5, b.solid(1, 1, 1), tex_img)),
        b.lambertian(b.noise(2.0)), b.metal([0.9, 0.8, 0.7], 0.3), b.dielectric(b.solid(0.9, 1.0, 0.9), 1.33),
        b.mix(white, b.metal([1, 1, 1], 0.0), 0.4), b.transparent(),
        b.portal([0.9, 0.9, 1.0], [0.0, 0.0, -6.0], b.quat_axis_angle([0, 1, 0], 20.0)),
        b.diffuse_light(b.solid(0.5, 0.4, 0.3), inner=white), b.isotropic(b.solid(0.5, 0.5, 0.9)),
    ]
    objs = []
    for k, m in enumerate(mats):
        x, y = (k % 4) * 2.2 - 3.3, (k // 4) * 2.2 - 2.0
        objs.append(b.sphere([x, y, 0], 1.0, m) if k % 2 == 0 else b.quad([x - 0.9, y - 0.9, 0], [1.8, 0, 0], [0, 1.8, 0], m))
    floor = b.quad([-8, -3.2, -8], [16, 0, 0], [0, 0, 16], white)
    light = b.diffuse_light(b.solid(10, 10, 10))
    q = b.quat_axis_angle([1, 0, 0], 25.0)
    l1 = b.transform(b.quad([-1, 0, -1], [2, 0, 0], [0, 0, 2], light), offset=[0, 6, 2], quat=q, scale=[1.5, 1.5, 1.5])
    l2 = b.triangle([3, 5, -1], [2, 0, 0], [0, 0, 2], light)
    world = b.list([b.bvh(objs), floor, l1, l2])
    e = b.empty()
    lights = b.list([b.transform(b.quad([-1, 0, -1], [2, 0, 0], [0, 0, 2], e), offset=[0, 6, 2], quat=q, scale=[1.5, 1.5, 1.5]),
                     b.list([b.triangle([3, 5, -1], [2, 0, 0], [0, 0, 2], e), b.sphere([-3.3, 0.2, 0], 1.0, e)])])  # the metal ball
    hs = b.finish(world, lights, width=48, spp=16, max_depth=10, vfov=50, look_from=(0, 1, 12), look_at=(0, 0, 0),
                  background=b.gradient([1, 1, 1], [0.5, 0.7, 1.0]), defocus_angle=0.8, focus_dist=12.0)
    hs._builder = b
    return hs


def disney_scene(rt, with_lights=True, width=64, spp=16, depth=8, seed=2):
    """Five Disney spheres covering every lobe + one with a base-colour image texture (obj.rs:271-293)."""
    rng = np.random.default_rng(seed)
    b = rt.Builder(seed)
    white = b.lambertian(b.solid(0.7, 0.7, 0.7))
    light = b.diffuse_light(b.solid(8, 8, 8))
    tex = b.image(rng.uniform(0.1, 1, (8, 16, 4)).astype(np.float32))
    mats = [b.disney((0.8, 0.3, 0.2), roughness=0.4),
            b.disney((0.9, 0.8, 0.3), metallic=1.0, roughness=0.3, anisotropic=0.5),
            b.disney((0.9, 0.9, 0.9), spec_trans=1.0, roughness=0.1, ior=1.5),
            b.disney((0.2, 0.4, 0.8), clearcoat=1.0, clearcoat_gloss=0.9, sheen=0.5, sheen_tint=0.5, roughness=0.6, specular_tint=0.3),
            b.disney((0.6, 0.8, 0.6), thin=1.0, flatness=0.5, diff_trans=0.5, spec_trans=0.3, roughness=0.5),
            b.disney((1, 1, 1), tex=tex, roughness=0.7, metallic=0.2, spec_trans=0.2, clearcoat=0.3)]
    objs = [b.quad([-9, -1, -8], [18, 0, 0], [0, 0, 16], white), b.quad([-2, 5, -2], [4, 0, 0], [0, 0, 4], light)]
    for k, m in enumerate(mats):
        objs.append(b.sphere([k * 2.2 - 5.5, 0, 0], 1.0, m))
    lights = b.list([b.quad([-2, 5, -2], [4, 0, 0], [0, 0, 4], b.empty())]) if with_lights else rt.RT_NONE
    hs = b.finish(b.list([b.bvh(objs)]), lights, width=width, aspect=2.0, spp=spp, max_depth=depth, vfov=38, look_from=(0, 3, 13),
                  look_at=(0, 0, 0), background=b.solid(0.1, 0.1, 0.15))
    hs._builder = b
    return hs


def obj_mesh_scene(rt, width=56, spp=16, depth=8, seed=3):
    """A small mesh built face by face the way shapes/obj.rs load_object does: every triangle carries its
    own RemappedMaterial (uv frame, smooth vertex normals, raw normal map), models in their own BVH."""
    rng = np.random.default_rng(seed)
    b = rt.Builder(seed)
    albedo = b.image(rng.uniform(0.2, 1, (16, 16, 4)).astype(np.float32))
    nm = rng.uniform(0.35, 0.65, (8, 8, 4)).astype(np.float32)
    nm[..., 2] = rng.uniform(0.8, 1.0, (8, 8))
    normal_map = b.image(nm, raw=True)
    alpha = rng.uniform(0, 1, (8, 8, 4)).astype(np.float32)
    alpha[..., 3] = (rng.uniform(0, 1, (8, 8)) > 0.3)
    alpha_tex = b.image(alpha)
    inner = [b.lambertian(albedo), b.disney((1, 1, 1), tex=albedo, roughness=0.4, metallic=0.3),
             b.diffuse_light(b.solid(0.4, 0.3, 0.2), inner=b.disney((0.7, 0.7, 0.9), roughness=0.5))]
    # Mix::from_image(Transparent, mat, alpha texture) as for `dissolve_texture` (obj.rs:318-325) and the
    # constant-ratio Mix of `dissolve < 1` (obj.rs:326-330)
    inner.append(b.mix_image(b.transparent(), inner[0], alpha_tex))
    inner.append(b.mix(b.transparent(), inner[1], 0.6))
    n = 6
    xs = np.linspace(-3, 3, n + 1)

    def height(x, z):
        return 0.4 * np.sin(1.3 * x) * np.cos(1.1 * z)

    def vertex(i, j):
        x, z = xs[i], xs[j]
        p = np.array([x, height(x, z), z])
        dx, dz = 0.4 * 1.3 * np.cos(1.3 * x) * np.cos(1.1 * z), -0.4 * 1.1 * np.sin(1.3 * x) * np.sin(1.1 * z)
        nrm = np.array([-dx, 1.0, -dz])
        return p, np.array([i / n, j / n]), nrm / np.linalg.norm(nrm)

    models = []
    for k, mat in enumerate(inner):
        faces = []
        for i in range(n):
            for j in range(n):
                if (i + j) % len(inner) != k:
                    continue
                quad = [vertex(i, j), vertex(i + 1, j), vertex(i + 1, j + 1), vertex(i, j + 1)]
                for tri in ((0, 1, 2), (0, 2, 3)):
                    pos = [quad[t][0] for t in tri]
                    uv = [quad[t][1] for t in tri]
                    nr = [quad[t][2] for t in tri]
                    f = b.obj_face(mat, pos, uv, nr, normal_map if k % 2 == 0 else rt.RT_NONE)
                    if f != rt.RT_NONE:
                        faces.append(f)
        models.append(b.bvh(faces))
    wavefont = b.list(models)
    light = b.quad([-2, 5, -2], [4, 0, 0], [0, 0, 4], b.diffuse_light(b.solid(9, 9, 9)))
    floor = b.quad([-8, -2, -8], [16, 0, 0], [0, 0, 16], b.lambertian(b.solid(0.6, 0.6, 0.6)))
    lights = b.list([b.quad([-2, 5, -2], [4, 0, 0], [0, 0, 4], b.empty())])
    hs = b.finish(b.list([wavefont, light, floor]), lights, width=width, spp=spp, max_depth=depth, vfov=40, look_from=(0, 5, 9), look_at=(0, 0, 0),
                  background=b.solid(0.15, 0.15, 0.2))
    hs._builder = b
    return hs


def write_synthetic_assets(root, n=24, seed=5):
    """A config-4-like asset directory: OBJ/MTL text + PNG textures, generated (no reference files)."""
    import os
    from PIL import Image
    rng = np.random.default_rng(seed)
    d = os.path.join(root, "Synth")
    os.makedirs(d, exist_ok=True)
    Image.fromarray((rng.uniform(0.2, 1, (32, 32, 3)) * 255).astype(np.uint8)).save(os.path.join(d, "albedo.png"))
    em = np.zeros((16, 16, 3), dtype=np.uint8)
    em[4:8, 4:12] = (255, 180, 60)
    Image.fromarray(em).save(os.path.join(d, "emit.png"))
    nm = (rng.uniform(0.4, 0.6, (16, 16, 3)) * 255).astype(np.uint8)
    nm[..., 2] = 255
    Image.fromarray(nm).save(os.path.join(d, "normal.png"))
    al = np.zeros((16, 16, 4), dtype=np.uint8)
    al[..., :3] = 255
    al[..., 3] = (rng.uniform(0, 1, (16, 16)) > 0.4) * 255
    Image.fromarray(al, "RGBA").save(os.path.join(d, "alpha.png"))
    with open(os.path.join(d, "terrain.mtl"), "w") as f:
        f.write("newmtl ground\nKd 0.8 0.8 0.8\nNi 1.45\nPr 0.7\nPm 0.0\nPc 0.2\nPcr 0.03\nmap_Kd albedo.png\nmap_Bump -bm 1.000000 normal.png\n\n"
                "newmtl glow\nKd 0.5 0.5 0.6\nNi 1.5\nPr 0.4\nPm 0.3\nmap_Ke emit.png\n\n"
                "newmtl leaves\nKd 0.2 0.7 0.3\nPr 0.6\nmap_d alpha.png\nd 0.8\nKe 0.0 0.1 0.0\n")
    xs = np.linspace(-4, 4, n + 1)
    with open(os.path.join(d, "terrain.obj"), "w") as f:
        f.write("mtllib terrain.mtl\no terrain\n")
        for j in range(n + 1):
            for i in range(n + 1):
                x, z = xs[i], xs[j]
                f.write(f"v {x:.6f} {0.5 * np.sin(x) * np.cos(0.8 * z):.6f} {z:.6f}\n")
        for j in range(n + 1):
            for i in range(n + 1):
                f.write(f"vt {i / n:.6f} {j / n:.6f}\n")
        for j in range(n + 1):
            for i in range(n + 1):
                x, z = xs[i], xs[j]
                nv = np.array([-0.5 * np.cos(x) * np.cos(0.8 * z), 1.0, 0.4 * np.sin(x) * np.sin(0.8 * z)])
                nv /= np.linalg.norm(nv)
                f.write(f"vn {nv[0]:.4f} {nv[1]:.4f} {nv[2]:.4f}\n")
        vid = lambda i, j: j * (n + 1) + i + 1
        for k, name in enumerate(["ground", "glow", "leaves"]):
            f.write(f"usemtl {name}\n")
            for j in range(n):
                for i in range(n):
                    if (i // 4 + j // 4) % 3 != k:
                        continue
                    a, b_, c, e = vid(i, j), vid(i + 1, j), vid(i + 1, j + 1), vid(i, j + 1)
                    f.write(f"f {a}/{a}/{a} {c}/{c}/{c} {b_}/{b_}/{b_}\nf {a}/{a}/{a} {e}/{e}/{e} {c}/{c}/{c}\n")
    # a glass ball (vanilla dielectric: Tf 1 1 1) and a closed fog shell, both UV spheres
    def uv_sphere(path, mtl, mat, centre, radius, seg):
        with open(path, "w") as f:
            f.write(f"mtllib {mtl}\no ball\n")
            for a in range(seg + 1):
                for b2 in range(2 * seg):
                    th, ph = np.pi * a / seg, np.pi * b2 / seg
                    nv = np.array([np.sin(th) * np.cos(ph), np.cos(th), np.sin(th) * np.sin(ph)])
                    p = centre + radius * nv
                    f.write(f"v {p[0]:.6f} {p[1]:.6f} {p[2]:.6f}\nvt {b2 / (2 * seg):.6f} {1 - a / seg:.6f}\nvn {nv[0]:.4f} {nv[1]:.4f} {nv[2]:.4f}\n")
            f.write(f"usemtl {mat}\n")
            vid2 = lambda a, b2: a * 2 * seg + (b2 % (2 * seg)) + 1
            for a in range(seg):
                for b2 in range(2 * seg):
                    q = [vid2(a, b2), vid2(a + 1, b2), vid2(a + 1, b2 + 1), vid2(a, b2 + 1)]
                    f.write("f " + " ".join(f"{v}/{v}/{v}" for v in q) + "\n")  # quads: exercises the fan triangulation
    with open(os.path.join(d, "ball.mtl"), "w") as f:
        f.write("newmtl glass\nKd 1.0 1.0 1.0\nNi 1.5\nTf 1.0 1.0 1.0\n")
    with open(os.path.join(d, "fog.mtl"), "w") as f:
        f.write("newmtl fog\nKd 1.0 1.0 1.0\n")
    uv_sphere(os.path.join(d, "ball.obj"), "ball.mtl", "glass", np.array([0.0, 1.6, 0.5]), 0.9, 8)
    uv_sphere(os.path.join(d, "fog.obj"), "fog.mtl", "fog", np.array([-1.5, 1.2, -1.0]), 1.4, 5)
    return root


def synthetic_obj_scene(rt, assets_root, width=64, spp=16, depth=10, seed=6):
    """The shape of obj_scene() (main.rs:207-382): Wavefont meshes, a fog mesh medium, a portal, transformed boards as
    lights, a thin translucent Disney board — built from generated assets through the Python OBJ loader."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("objload", os.path.join(os.path.dirname(rt.__file__), "objload.py"))
    objload = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(objload)
    b = rt.Builder(seed)
    wf = objload.Wavefont(b, assets_root)
    terrain = wf.new("terrain.obj", "Synth", False)
    ball = wf.new("ball.obj", "Synth", True)
    fog = b.medium(wf.new("fog.obj", "Synth", False), 0.6, b.solid(1.0, 0.936, 0.381))
    portal = b.quad([-3.5, 0.2, -3.0], [1.5, 0, -0.5], [0, 2.5, 0], b.portal([1, 1, 1], [5.0, 0.0, 2.0], [1, 0, 0, 0]))
    trans = b.transform(b.quad([-1, 0, -1], [0, 0, 2], [2, 0, 0], b.disney((0.8, 0.8, 0.8), diff_trans=1.0, roughness=1.0, thin=1.0)),
                        offset=[2.5, 1.5, -2.0], quat=b.quat_axis_angle([0.993, -0.082, 0.082], 90.4), scale=[1.6, 1.0, 1.0])
    def board(mat, off, axis, deg, s):
        return b.transform(b.quad([-1, 0, -1], [0, 0, 2], [2, 0, 0], mat), offset=off, quat=b.quat_axis_angle(axis, deg), scale=[s, s, s])
    l1 = ([-0.4, 5.3, 0.9], [0.921, 0.021, 0.389], 34.7, 2.0)
    l2 = ([-3.0, 2.5, 2.5], [0.766, 0.483, -0.423], 85.7, 0.8)
    world = b.list([terrain, board(b.diffuse_light(b.solid(6, 6, 6)), *l1), ball, trans, portal,
                    board(b.diffuse_light(b.solid(5.0, 3.4, 0.0)), *l2), fog])
    lights = b.list([board(b.empty(), *l1), board(b.empty(), *l2)])
    hs = b.finish(world, lights, width=width, aspect=16 / 9, spp=spp, max_depth=depth, vfov=35, look_from=(0.5, 4.0, 9.5), look_at=(0, 0.8, 0),
                  background=b.gradient([0.6, 0.6, 0.7], [0.2, 0.3, 0.6]))
    hs._builder = b
    return hs
