"""The lean variants of the shade-class kernels (scene_types.h, ShadeLean): a scene whose light list is flat, short and untransformed
shades its diffuse and textured hits against a light list staged in shared memory; its isotropic class takes a fog's scatter point
without the Transform, texture and HitRecord code when every thin medium is untransformed with a solid albedo; its emissive class
only adds the light's colour when every light surface is untransformed with a solid colour.  The draws are addressed, so the image,
the segment count and the error count must be those of the general kernel (binning switched off); a scene that misses a condition
keeps the general kernel of the classes that condition concerns."""
import pytest

from test_gpu_parity import image_close

ALL = "diffuse textured isotropic emissive"


def lean_scene(rt, variant):
    """book2's situation in small: a quad light in a flat list, a thin fog around everything, a thick ball with its glass shell,
    solid and checker-textured Lambertians, some of them below a Transform."""
    b = rt.Builder(5)
    checker = b.checker(0.5, b.solid(0.3, 0.5, 0.9), b.solid(0.9, 0.5, 0.3))
    floor = b.quad([-6, -1.5, -6], [12, 0, 0], [0, 0, 12], b.lambertian(b.solid(0.6, 0.6, 0.6)))
    # the lamp's plane y = 4 must not lie on a checker boundary (floor(scale * y) would decide on rounding)
    lamp_tex = b.checker(0.7, b.solid(12, 12, 12), b.solid(4, 4, 4)) if variant == "checker_lamp" else b.solid(12, 12, 12)
    lamp = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.diffuse_light(lamp_tex))
    light_quad = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.empty())
    fog_albedo = checker if variant == "checker_fog" else b.solid(1, 1, 1)
    fog = b.medium(b.sphere([0, 0, 0], 30.0, b.empty()), 0.01, fog_albedo)
    if variant == "fog_xform":
        fog = b.transform(fog, offset=[0.1, 0, 0])
    thick = b.medium(b.sphere([0, 0, 0], 1.0, b.empty()), 6.0, b.solid(0.3, 0.5, 0.9))
    shell = b.sphere([0, 0, 0], 1.0, b.dielectric(b.solid(1, 1, 1), 1.5))
    ball = b.sphere([2.2, -0.9, 0.8], 0.6, b.lambertian(checker))
    moved = b.transform(b.sphere([0, 0, 0], 0.5, b.lambertian(b.solid(0.8, 0.3, 0.2))), offset=[-2.2, -1.0, 0.6])
    if variant == "lamp_xform":  # the lamp's surface below a Transform; the light list keeps its untransformed quad
        lamp = b.transform(lamp, offset=[0.1, 0.0, 0.0])
    lights = [light_quad]
    if variant == "light_xform":  # the light list's quad below a Transform; the lamp itself stays as it is
        lights = [b.transform(light_quad, offset=[0.1, 0.0, 0.0])]
    elif variant == "five_lights":
        lights += [b.sphere([-3.0 + 1.5 * k, 3.0, -2.0], 0.2, b.empty()) for k in range(4)]
    elif variant == "nested_lights":  # weights 1/2, 1/4, 1/4: not a flat list
        lights.append(b.list([b.sphere([-2.0, 3.0, -2.0], 0.2, b.empty()), b.sphere([2.0, 3.0, -2.0], 0.2, b.empty())]))
    things = [floor, lamp, fog, thick, shell, ball, moved]
    return b.finish(b.list(things), b.list(lights), width=40, spp=16, max_depth=24, vfov=35, look_from=(0, 1.5, 6),
                    background=b.solid(0.5, 0.6, 0.8))


LEAN = {
    "book2": ALL,
    "light_xform": "emissive",
    "five_lights": "emissive",
    "nested_lights": "emissive",
    "fog_xform": "diffuse textured emissive",
    "checker_fog": "diffuse textured emissive",
    "lamp_xform": "diffuse textured isotropic",
    "checker_lamp": "diffuse textured isotropic",
}


def _shade_choice(rt, hs, monkeypatch, capfd):
    """The scene compiler's choice, as it reports it (RT2025_TIMING); rt_scene_create needs no device up to that point."""
    monkeypatch.setenv("RT2025_TIMING", "1")
    capfd.readouterr()
    try:
        rt.Scene(hs)
    except Exception:
        pass  # no device here: the scene was compiled before the device check failed
    err = capfd.readouterr().err
    lines = [l for l in err.splitlines() if "[rt2025 compile] shade lean:" in l]
    assert len(lines) == 1, err
    return lines[0].split("shade lean: ")[1].strip()


@pytest.mark.parametrize("variant", sorted(LEAN))
def test_shade_lean_eligibility(rt, variant, monkeypatch, capfd):
    assert _shade_choice(rt, lean_scene(rt, variant), monkeypatch, capfd) == LEAN[variant]


def test_shade_lean_book2_eligibility(rt, monkeypatch, capfd):
    hs = rt.named_scene("book2_final", seed=7, params=[40, 9, 40])
    assert _shade_choice(rt, hs, monkeypatch, capfd) == ALL


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(LEAN))
def test_shade_lean_vs_general_kernel_and_oracle(gpu, rt, orc, variant, monkeypatch):
    hs = lean_scene(rt, variant)
    monkeypatch.setenv("RT2025_TAIL_PATHS", "0")  # these frames are small enough for k_tail to finish them after one iteration
    a, sa = rt.Scene(hs).render(seed=9)
    assert sa.shade_lean_hits > 0
    c, sc_ = rt.Scene(hs).render(seed=9, no_binning=True)  # every hit through the general k_shade<SC_OTHER>
    assert sc_.shade_lean_hits == 0
    assert sa.segments == sc_.segments and sa.errors == sc_.errors
    image_close(a, c, frac_bad=0.0, rel=1e-9)
    ref, _ = orc.OracleScene(hs).render(seed=9)
    image_close(a, ref)


@pytest.mark.gpu
def test_shade_lean_runs_on_book2(gpu, rt, monkeypatch):
    monkeypatch.setenv("RT2025_TAIL_PATHS", "0")  # a frame this small is otherwise finished by k_tail after one iteration
    hs = rt.named_scene("book2_final", seed=7, params=[40, 9, 40])
    _, st = rt.Scene(hs).render(seed=5)
    assert st.shade_lean_hits > 0
