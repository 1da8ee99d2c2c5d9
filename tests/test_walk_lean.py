"""The lean variant of the random-walk kernel (scene_types.h, WalkLean): scenes whose walk needs no Transform, texture lookup or
light-tree code run a k_walk with the walk's constants staged in shared memory, and the glass shell that shares the thick
medium's boundary sphere takes its hit from the boundary test's roots.  The draws are addressed, so the image, the segment
count and the error count must be those of the plain wavefront (walk switched off); scenes that miss one condition keep the
generic kernel."""
import numpy as np
import pytest

from test_gpu_parity import _walk_scene, image_close


def lean_scene(rt, variant):
    """book2's situation in small: a thick ball with its glass shell in the world, a thin fog around everything, a quad light."""
    b = rt.Builder(5)
    floor = b.quad([-6, -1.5, -6], [12, 0, 0], [0, 0, 12], b.lambertian(b.solid(0.6, 0.6, 0.6)))
    lamp = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.diffuse_light(b.solid(12, 12, 12)))
    light_quad = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.empty())
    albedo = b.checker(0.5, b.solid(0.3, 0.5, 0.9), b.solid(0.9, 0.5, 0.3)) if variant == "textured" else b.solid(0.3, 0.5, 0.9)
    thick = b.medium(b.sphere([0, 0, 0], 1.0, b.empty()), 6.0, albedo)
    fog = b.medium(b.sphere([0, 0, 0], 30.0, b.empty()), 0.01, b.solid(1, 1, 1))
    glass = b.dielectric(b.solid(1, 1, 1), 1.5)
    shell = b.sphere([0, 0, 0], 1.0, glass)
    things = [floor, lamp, thick, fog]
    lights = [light_quad]
    if variant == "two_lights":  # a quad and a sphere in the flat light list
        things += [shell, b.sphere([2.5, 3.0, 0.5], 0.4, b.diffuse_light(b.solid(8, 6, 4)))]
        lights.append(b.sphere([2.5, 3.0, 0.5], 0.4, b.empty()))
    elif variant == "no_shell":  # the entry leaf holds an unrelated primitive inside the ball
        things.append(b.sphere([0.2, 0.1, 0.0], 0.3, b.lambertian(b.solid(0.8, 0.2, 0.2))))
    elif variant == "shell_shared":  # the shell shares its leaf with a quad inside the ball
        things += [shell, b.quad([-0.5, -0.3, -0.4], [0.6, 0, 0], [0, 0.5, 0.3], b.lambertian(b.solid(0.8, 0.2, 0.2)))]
    elif variant == "shell_ulp":  # a shell one ulp larger than the boundary: no shortcut, its own sphere test
        things.append(b.sphere([0, 0, 0], float(np.nextafter(1.0, 2.0)), glass))
    elif variant == "light_xform":  # the light (and the lamp) below a Transform
        things[1] = b.transform(lamp, offset=[0.1, 0, 0])
        lights = [b.transform(light_quad, offset=[0.1, 0, 0])]
    elif variant == "two_thick":  # a second thick medium
        things += [shell, b.medium(b.sphere([2.5, 0, 0], 0.8, b.empty()), 4.0, b.solid(0.9, 0.4, 0.3))]
    else:  # "book2", "textured"
        things.append(shell)
    return b.finish(b.list(things), b.list(lights), width=40, spp=16, max_depth=24, vfov=35, look_from=(0, 1.5, 6),
                    background=b.solid(0.5, 0.6, 0.8))


LEAN = {"book2": "lean, shell", "two_lights": "lean, shell", "no_shell": "lean", "shell_shared": "lean, shell", "shell_ulp": "lean",
        "light_xform": "generic", "textured": "generic", "two_thick": "generic"}
# test_gpu_parity's walk scenes: "surfaces_inside" (a metal ball, a quad and the glass shell inside the boundary, one quad light)
# meets every condition, so its parity test checks the lean kernel; the three others keep the generic one
EXISTING = {"surfaces_inside": "lean, shell", "overlapping": "generic", "many_neighbours": "generic", "moving_transformed": "generic"}


def _walk_choice(rt, hs, monkeypatch, capfd):
    """The scene compiler's choice, as it reports it (RT2025_TIMING); rt_scene_create needs no device up to that point."""
    monkeypatch.setenv("RT2025_TIMING", "1")
    capfd.readouterr()
    try:
        rt.Scene(hs)
    except Exception:
        pass  # no device here: the scene was compiled before the device check failed
    err = capfd.readouterr().err
    lines = [l for l in err.splitlines() if "[rt2025 compile] random walk:" in l]
    assert len(lines) == 1, err
    return lines[0].split("random walk: ")[1].strip()


@pytest.mark.parametrize("variant", sorted(LEAN))
def test_walk_lean_eligibility(rt, variant, monkeypatch, capfd):
    assert _walk_choice(rt, lean_scene(rt, variant), monkeypatch, capfd) == LEAN[variant]


@pytest.mark.parametrize("variant", sorted(EXISTING))
def test_walk_lean_existing_walk_scenes(rt, variant, monkeypatch, capfd):
    assert _walk_choice(rt, _walk_scene(rt, variant), monkeypatch, capfd) == EXISTING[variant]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(LEAN))
def test_walk_lean_vs_wavefront_and_oracle(gpu, rt, orc, variant, monkeypatch):
    hs = lean_scene(rt, variant)
    monkeypatch.setenv("RT2025_TAIL_PATHS", "0")  # these frames are small enough for k_tail to finish them after one iteration
    a, sa = rt.Scene(hs).render(seed=9)
    assert sa.walk_segments > 0
    assert sa.walk_lean_segments == (sa.walk_segments if LEAN[variant] != "generic" else 0)
    monkeypatch.setenv("RT2025_WALK_DRAIN_QUEUE", "0")  # walks of any length
    a2, sa2 = rt.Scene(hs).render(seed=9)
    monkeypatch.delenv("RT2025_WALK_DRAIN_QUEUE")
    assert sa2.walk_segments > sa.walk_segments
    monkeypatch.setenv("RT2025_WALK_MIN_DEPTH", "0")
    c, sc_ = rt.Scene(hs).render(seed=9)
    monkeypatch.delenv("RT2025_WALK_MIN_DEPTH")
    assert sc_.walk_segments == 0
    assert sa.segments == sa2.segments == sc_.segments and sa.errors == sa2.errors == sc_.errors
    image_close(a, c, frac_bad=0.0, rel=1e-9)
    image_close(a2, c, frac_bad=0.0, rel=1e-9)
    ref, _ = orc.OracleScene(hs).render(seed=9)
    image_close(a, ref)


@pytest.mark.gpu
def test_walk_lean_runs_on_book2(gpu, rt, monkeypatch):
    monkeypatch.setenv("RT2025_TAIL_PATHS", "0")  # a frame this small is otherwise finished by k_tail after one iteration
    hs = rt.named_scene("book2_final", seed=7, params=[40, 9, 40])
    _, st = rt.Scene(hs).render(seed=5)
    assert st.walk_segments > 0 and st.walk_lean_segments == st.walk_segments
