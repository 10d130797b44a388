"""GPU tests of the reference-facing Python API (the drop-in boundary): Ray / Intersection, the render entry points,
and RayTracerEnv (scalar and batched), all through the C ABI, against golden vectors recorded from the unmodified
reference and against the oracle."""
import numpy as np
import pytest

from conftest import gate, load_golden

pytestmark = pytest.mark.gpu

ENVS = ["env_rl_optimized", "env_rl_demo", "env_fb_demo", "env_fb_balls", "env_rl_balls_rotated", "env_rl_adaptive"]


def make_env(rt, z, fs, B, precision):
    from ray_tracer_v1_b200.ray_tracer_env import BatchedRayTracerEnv
    return BatchedRayTracerEnv(fs, B, int(z["width"]), int(z["height"]), camera_position=tuple(z["cam"]),
                               camera_angle=tuple(z["cam_angle"]), fov=float(z["fov"]), max_bounces=int(z["max_bounces"]),
                               flavour=str(z["flavour"]), precision=precision,
                               reward_mode="adaptive" if "adaptive" in str(z.get("name", "")) else "default")


@pytest.mark.parametrize("name", ENVS)
def test_batched_env_matches_reference_rollouts(rt, name):
    """Rollouts recorded from the UNMODIFIED reference env (96 episodes x T steps, stepping on past termination)."""
    z, fs = load_golden(name)
    z["name"] = name
    B = z["pixels"].shape[0]
    env = make_env(rt, z, fs, B, "f64")
    obs0, _ = env.reset(options={"pixels": z["pixels"]})
    np.testing.assert_allclose(obs0.cpu().numpy(), z["obs0"], rtol=1e-6, atol=1e-7)
    # the reference feeds float32 actions into numpy trig, so part of ITS arithmetic is float32 (see test_oracle_golden)
    for t in range(z["actions"].shape[0]):
        obs, rew, term, trunc, info = env.step(z["actions"][t])
        np.testing.assert_allclose(obs.cpu().numpy(), z["obs"][t], rtol=5e-5, atol=5e-6, err_msg=f"obs step {t}")
        np.testing.assert_allclose(rew.cpu().numpy(), z["reward"][t], rtol=1e-5, atol=1e-6, err_msg=f"reward step {t}")
        assert np.array_equal(term.cpu().numpy(), z["terminated"][t].astype(bool))
        assert np.array_equal(trunc.cpu().numpy(), z["truncated"][t].astype(bool))
        assert np.array_equal(info["reason"].cpu().numpy(), z["reason"][t])
        np.testing.assert_allclose(info["total_reward"].cpu().numpy(), z["total_reward"][t], rtol=1e-5, atol=1e-5)
    env.close()


@pytest.mark.parametrize("name", ENVS)
def test_batched_env_fp64_equals_oracle_and_fp32_is_close(rt, orc, name):
    z, fs = load_golden(name)
    z["name"] = name
    B = z["pixels"].shape[0]
    ref = orc.OracleEnv(fs, B, int(z["width"]), int(z["height"]), camera=z["cam"], camera_angle=z["cam_angle"],
                        fov=float(z["fov"]), max_bounces=int(z["max_bounces"]), flavour=str(z["flavour"]),
                        adaptive="adaptive" in name)
    e64, e32 = make_env(rt, z, fs, B, "f64"), make_env(rt, z, fs, B, "f32")
    o_ref = ref.reset(z["pixels"])
    o64, _ = e64.reset(options={"pixels": z["pixels"]})
    o32, _ = e32.reset(options={"pixels": z["pixels"]})
    np.testing.assert_allclose(o64.cpu().numpy(), o_ref, rtol=1e-6, atol=1e-7)
    alive32 = np.ones(B, bool)                      # FP32 episodes that still follow the FP64 trajectory
    for t in range(z["actions"].shape[0]):
        a = z["actions"][t]
        obs_r, rew_r, term_r, trunc_r, reason_r = ref.step(a)
        obs, rew, term, trunc, info = e64.step(a)
        np.testing.assert_allclose(obs.cpu().numpy(), obs_r, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(rew.cpu().numpy(), rew_r, rtol=1e-9, atol=1e-12)
        assert np.array_equal(term.cpu().numpy(), term_r) and np.array_equal(trunc.cpu().numpy(), trunc_r)
        assert np.array_equal(info["reason"].cpu().numpy(), reason_r)
        obs3, rew3, term3, trunc3, info3 = e32.step(a)
        same = info3["reason"].cpu().numpy() == reason_r
        alive32 &= same                              # a flipped hit/miss sends an episode down another path: drop it
        ok = alive32
        np.testing.assert_allclose(obs3.cpu().numpy()[ok], obs_r[ok], rtol=2e-3, atol=2e-3)
        np.testing.assert_allclose(rew3.cpu().numpy()[ok], rew_r[ok], rtol=2e-3, atol=6e-3)
    gate(f"{name} FP32 episodes leaving the FP64 trajectory", 1 - alive32.mean(), 2.5 / B)       # measured 0 of 96 (65,536 envs: 5.5e-4)
    e64.close(); e32.close()


def test_scalar_env_dropin(rt):
    """The scalar RayTracerEnv keeps the reference's return types and info keys."""
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.ray_tracer_env import RayTracerEnv, FBRayTracerEnv
    from ray_tracer_v1_b200 import Vector, Colour
    z, fs = load_golden("env_rl_optimized")
    spec = scenes.build_optimized_env_scene()
    env = RayTracerEnv(spheres=spec.spheres, image_width=320, image_height=240, camera_position=Vector(0, 0, 0), fov=80,
                       max_bounces=6, background_colour=Colour(0, 0, 0), point_light_sources=spec.point_lights)
    for b in (0, 3, 17):
        px = tuple(int(v) for v in z["pixels"][b])
        obs, info = env.reset(options={"pixel": px})
        assert obs.shape == (18,) and obs.dtype == np.float32 and info["pixel"] == px and "initial_ray" in info
        np.testing.assert_allclose(obs, z["obs0"][b], rtol=1e-6, atol=1e-7)
        for t in range(4):
            obs, reward, terminated, truncated, info = env.step(z["actions"][t, b])
            assert isinstance(reward, float) and isinstance(terminated, bool) and isinstance(truncated, bool)
            np.testing.assert_allclose(obs, z["obs"][t, b], rtol=5e-5, atol=5e-6)
            np.testing.assert_allclose(reward, z["reward"][t, b], rtol=1e-5, atol=1e-6)
            assert terminated == bool(z["terminated"][t, b])
            assert {"bounce_count", "through_count", "total_reward"} <= set(info)
    env.close()
    fb = FBRayTracerEnv(spheres=scenes.build_balls_in_space(as_rendered=False).spheres, image_width=160, image_height=120,
                        camera_position=Vector(0, 0, 1), fov=60, max_bounces=5)
    obs, _ = fb.reset(options={"pixel": (80, 60)})
    obs, reward, terminated, truncated, info = fb.step(fb.action_space.sample())
    assert obs.shape == (18,)
    fb.close()


def test_batched_env_c5_size_and_sharding(rt):
    """BASELINE config 5: 65,536 parallel envs; env shards are independent, so a shard equals the same rows of the whole."""
    import torch
    from ray_tracer_v1_b200 import scenes, flatten_scene
    from ray_tracer_v1_b200.ray_tracer_env import BatchedRayTracerEnv
    from ray_tracer_v1_b200.distributed import env_slices
    spec = scenes.build_balls_in_space(as_rendered=False)
    fs = flatten_scene(spec.spheres, spec.global_lights, [], spec.background)
    B = 65536
    kw = dict(image_width=320, image_height=240, camera_position=(0, 0, 1), fov=60, max_bounces=5, flavour="fb")
    rs = np.random.RandomState(0)
    pixels = np.stack([rs.randint(0, 320, B), rs.randint(0, 240, B)], 1).astype(np.int32)
    actions = rs.uniform(-1, 1, (6, B, 2)).astype(np.float32)
    whole = BatchedRayTracerEnv(fs, B, **kw)
    o, _ = whole.reset(options={"pixels": pixels})
    b0, b1 = env_slices(B, 8)[3]
    part = BatchedRayTracerEnv(fs, b1 - b0, **kw)
    op, _ = part.reset(options={"pixels": pixels[b0:b1]})
    assert torch.equal(o[b0:b1], op)
    done = torch.zeros(B, dtype=torch.bool, device="cuda")
    for t in range(6):
        o, r, te, tr, info = whole.step(torch.as_tensor(actions[t], device="cuda"))
        op, rp, tep, trp, _ = part.step(actions[t, b0:b1])
        assert torch.equal(o[b0:b1], op) and torch.equal(r[b0:b1], rp) and torch.equal(te[b0:b1], tep)
        done |= te
    assert bool(done.all())                       # every episode ends within max_bounces + 1 steps
    # device-drawn start pixels are reproducible and inside the image
    whole._resets = 0
    o1, i1 = whole.reset(seed=11)
    p1, o1 = i1["pixels"].clone(), o1.clone()
    whole._resets = 0
    o2, i2 = whole.reset(seed=11)
    assert torch.equal(p1, i2["pixels"]) and torch.equal(o1, o2)
    assert int(p1[:, 0].max()) < 320 and int(p1[:, 1].max()) < 240 and int(p1.min()) >= 0
    # env-sharded rollouts: a shard draws the start pixels of its GLOBAL env indices, so with device-drawn pixels and
    # the in-launch restarts of step_auto it still reproduces the same rows of the unsharded batch, step after step
    shard = BatchedRayTracerEnv.shard(fs, B, rank=3, world=8, **kw)
    whole._resets = 0
    ow, _ = whole.reset(seed=11)
    osh, _ = shard.reset(seed=11)
    assert torch.equal(ow[b0:b1], osh)
    for t in range(8):
        a = torch.as_tensor(actions[t % 6], device="cuda")
        o, r, te, tr, info = whole.step_auto(a)
        o2, r2, te2, tr2, info2 = shard.step_auto(a[b0:b1])
        assert torch.equal(o[b0:b1], o2) and torch.equal(r[b0:b1], r2) and torch.equal(te[b0:b1], te2)
        assert torch.equal(info["pixels"][b0:b1], info2["pixels"])
    whole.close(); part.close(); shard.close()


def test_ray_and_intersection_dropin(rt):
    """Notebook-style scalar calls: RL/Marbles 1.ipynb cell 7 and a terminalRGB round trip against the frame golden."""
    from ray_tracer_v1_b200 import Ray, Vector, Sphere, Material, scenes
    hit = Ray(Vector(0.1, 0, 5), Vector(0, 0, -1)).sphereDiscriminant(Sphere(Vector(0, 0, 0), 1, Material()))
    assert hit.intersects and hit.point.getXYZ() == (0.1, 0.0, 0.9949874371066194)
    z, fs = load_golden("whitted_c1_balls_320x240")
    spec = scenes.build_balls_in_space(as_rendered=True)
    cam = Vector(*spec.camera)
    for (yi, xi) in ((120, 160), (60, 100), (200, 250), (10, 10), (150, 40)):
        d = Vector(float(z["X"][xi]), float(z["Y"][yi]), -1).normalise()
        t = Ray(cam, d).nearestSphereIntersect(spec.spheres, max_bounces=1)
        if z["hit"][yi, xi] < 0:
            assert t is None
            continue
        assert t.object is spec.spheres[int(z["hit"][yi, xi])]
        c = t.terminalRGB(spheres=spec.spheres, background_colour=spec.background, global_light_sources=spec.global_lights,
                          point_light_sources=spec.point_lights)
        assert c.getList() == [float(v) for v in z["rgb"][yi, xi]]


def test_render_entry_points(rt, orc):
    from ray_tracer_v1_b200 import scenes, Vector
    from ray_tracer_v1_b200.renderers import (TraditionalRenderer, ComplexTraditionalRenderer, CustomSceneExperiment)
    import tempfile
    # output5: render_custom_scene('traditional') reproduces the reference's own 320x240 image
    z, _ = load_golden("whitted_c1_balls_320x240")
    with tempfile.TemporaryDirectory() as tmp:
        exp = CustomSceneExperiment(output_dir=tmp, precision="f64")
        exp.config.update(image_width=320, image_height=240, samples_per_pixel=1, max_bounces=1)
        t, img = exp.render_custom_scene(scenes.build_balls_in_space(as_rendered=False).spheres, "traditional", None)
        assert np.array_equal(img, z["image"]) and t > 0
        exp32 = CustomSceneExperiment(output_dir=tmp, precision="f32")
        exp32.config.update(image_width=320, image_height=240, samples_per_pixel=1, max_bounces=1)
        _, img32 = exp32.render_custom_scene(scenes.build_balls_in_space(as_rendered=False).spheres, "traditional", None)
        gate("render entry FP32 pixels beyond 1/255", (np.abs(img32 - z["image"]).max(axis=2) > 1.001 / 255).mean(), 1e-4)      # measured 0
        # the scalar helper behind the frame (RL/output5.py:535-607): the same pixels of the reference's image, one ray each
        from ray_tracer_v1_b200 import Ray
        balls = scenes.build_balls_in_space(as_rendered=False).spheres
        for (yi, xi) in ((120, 160), (60, 100), (200, 250), (10, 10), (150, 40)):
            ray = Ray(Vector(0, 0, 1), Vector(float(z["X"][xi]), float(z["Y"][yi]), -1).normalise())
            colour, stats, strategies = exp._trace_custom_traditional(ray, balls, 0)
            assert colour.getList() == [float(v) for v in z["rgb"][yi, xi]] and strategies == ['traditional_mimic']
            assert stats['light_hits'] == int(sum(colour.getList()) / 3 > 10)
        # an unchanged scene list is not uploaded again (content key), a mutated one is: same image twice, then the image
        # a fresh experiment renders of the mutated list
        _, again = exp.render_custom_scene(balls, "traditional", None)
        assert np.array_equal(again, z["image"]) and exp._context().h2d_bytes == 0
        balls[1].centre = Vector(0.4, 0.1, -2.5)
        _, moved = exp.render_custom_scene(balls, "traditional", None)
        assert exp._context().h2d_bytes > 0 and not np.array_equal(moved, z["image"])
        fresh = CustomSceneExperiment(output_dir=tmp, precision="f64")
        fresh.config.update(image_width=320, image_height=240, samples_per_pixel=1, max_bounces=1)
        assert np.array_equal(fresh.render_custom_scene(balls, "traditional", None)[1], moved)
        # render_true_original: 601x601 notebook grid; compare its centre crop rows with the 121-grid golden's geometry
        full = exp.render_true_original(scenes.build_balls_in_space(as_rendered=False).spheres, None)
        assert full.shape == (601, 601, 3) and full.max() <= 1.0 and full.min() >= 0.0
    # TraditionalRenderer: attribute injection like the reference's main(), stats keys, image == oracle render
    spec = scenes.build_chandelier()
    r = TraditionalRenderer(precision="f64", seed=5)
    r.scene = spec.spheres
    r.light_sources = [s for s in spec.spheres if s.material.emitive]
    r.small_lights = [s for s in r.light_sources if s.radius < 0.5]
    r.camera_position = Vector(0, 2, 0)
    img = r.render(64, 36, samples_per_pixel=3, max_bounces=8)
    sums, st = orc.render_path(r.flat_scene(), (0, 2, 0), 64, 36, 3, 8, 0.0, seed=5)
    assert np.array_equal(img, orc.resolve(sums, 3))
    assert r.stats["total_rays"] == st["total_rays"] and r.stats["light_hits"] == st["light_hits"]
    # trace_ray_traditional (the scalar recursive tracer, FB/fb_vs_traditional_chandelier.py:431-521) through
    # rt_trace_paths: fed the camera ray of a pixel sample (jitter = the Philox numbers render() uses) it reproduces that
    # sample, so the samples of a pixel add up to the frame's sum -- exactly, in the FP64 build
    for (x, y) in ((10, 20), (33, 5), (63, 35), (0, 0)):
        tot = np.zeros(3)
        for smp in range(3):
            u0, u1 = orc.rng_pair(5, y * 64 + x, smp, 0)
            ray = r.generate_camera_ray(x, y, 0.5 + (u0 - 0.5), 0.5 + (u1 - 0.5))
            tot += r.trace_ray_traditional(ray, 0, pixel=y * 64 + x, sample=smp).getList()
        assert np.array_equal(tot, sums[y, x]), (x, y, tot, sums[y, x])
    assert r.trace_ray_traditional(ray, bounce_count=8).getList() == [2.0, 2.0, 5.0]      # at the depth limit: Colour(2, 2, 5)
    # generate_camera_ray: the reference's camera (aspect applied twice on x), same direction as the device generates
    ray = r.generate_camera_ray(10, 20, 0.5, 0.5)
    hh = np.tan(np.radians(60) / 2)
    d = np.array([(2 * 10.5 / 64 - 1) * (64 / 36) * hh * (64 / 36), (1 - 2 * 20.5 / 36) * hh, -1.0])
    np.testing.assert_allclose(ray.D.getXYZ(), d / np.linalg.norm(d), rtol=1e-12)
    assert r.stats["rays_per_second"] > 0 and set(r.stats) == {'total_rays', 'total_intersections', 'light_hits',
                                                              'small_light_hits', 'render_time', 'rays_per_second'}
    spec.spheres[10].centre = Vector(0.3, 3.0, 7.0)          # scenes are mutable: the next render must see the change
    img2 = r.render(64, 36, samples_per_pixel=3, max_bounces=8)
    sums2, _ = orc.render_path(r.flat_scene(), (0, 2, 0), 64, 36, 3, 8, 0.0, seed=5)
    assert np.array_equal(img2, orc.resolve(sums2, 3)) and not np.array_equal(img, img2)
    c = ComplexTraditionalRenderer(precision="f32", seed=1)
    cs = scenes.build_complex()
    c.scene, c.light_sources = cs.spheres, [s for s in cs.spheres if s.material.emitive]
    c.small_lights = [s for s in c.light_sources if s.radius < 0.5]
    im = c.render(96, 54, samples_per_pixel=2, max_bounces=5)
    assert im.shape == (54, 96, 3) and im.dtype == np.float32 and 5.0 < c.stats["total_rays"] / (96 * 54 * 2) <= 6.0


def test_fb_trajectories_match_reference(rt, orc):
    """rt_generate_trajectories vs the reference-generated golden walks (FP64: same path, observations to float32
    rounding of a 1-ulp libm difference) and vs the oracle at a larger batch; FP32: same walk for most trajectories."""
    from conftest import gate, load_golden
    from ray_tracer_v1_b200 import fb_trajectories as fbt
    z, fs = load_golden("traj_complex_256")
    S, mb, seed = int(z["max_steps"]), int(z["max_bounces"]), int(z["seed"])
    b = fbt.generate_trajectories(fs, 256, S, mb, seed, precision="f64")
    assert np.array_equal(b.length.cpu().numpy(), z["length"]) and np.array_equal(b.hit_light.cpu().numpy(), z["hit_light"].astype(bool))
    assert np.array_equal(b.hit.cpu().numpy(), z["hit"].astype(bool)) and np.array_equal(b.reward.cpu().numpy(), z["reward"])
    for k, t in (("obs", b.obs), ("action", b.action), ("next_obs", b.next_obs)):
        np.testing.assert_allclose(t.cpu().numpy(), z[k], rtol=2e-6, atol=2e-6, err_msg=k)
    j = int(np.argmax(z["length"]))
    tr = b.transitions(j)
    assert len(tr) == int(z["length"][j]) > 0 and tr[0][0].shape == (22,) and tr[0][1].shape == (2,)
    big = fbt.generate_trajectories(fs, 20000, S, mb, seed + 1, precision="f64")
    ref = orc.generate_trajectories(fs, 20000, S, mb, seed + 1)
    assert np.array_equal(big.length.cpu().numpy(), ref["length"]) and np.array_equal(big.hit_light.cpu().numpy(), ref["hit_light"].astype(bool))
    np.testing.assert_allclose(big.next_obs.cpu().numpy(), ref["next_obs"], rtol=2e-6, atol=2e-6)
    f32 = fbt.generate_trajectories(fs, 20000, S, mb, seed + 1, precision="f32")
    same = f32.length.cpu().numpy() == ref["length"]
    assert same.mean() > 0.97
    # FP32 rounding is amplified at every bounce off a curved surface: the first transition is tight, the whole
    # walk (up to 8 bounces) stays close for most trajectories
    d = np.abs(f32.next_obs.cpu().numpy()[same] - ref["next_obs"][same])
    assert (d[:, 0].max(axis=1) < 2e-3).mean() > 0.97
    assert (d.max(axis=(1, 2)) < 5e-2).mean() > 0.9
    o, a, no, r, h = f32.flat()
    assert o.shape[0] == int(f32.length.sum()) and f32.queries >= o.shape[0]
    one, lit = fbt.generate_trajectory(fs, S, mb, seed=seed + 1)
    assert isinstance(lit, bool) and len(one) == int(f32.length[0])


def test_vec_env_adapter(rt):
    """RayTracerVecEnv: the SB3 VecEnv protocol over the batched env -- auto-reset of finished episodes with
    terminal_observation / TimeLimit.truncated, numpy and torch modes stepping the same episodes."""
    import torch
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.ray_tracer_env import RayTracerVecEnv, AdaptiveRewardRayTracerEnv
    spec = scenes.build_optimized_env_scene()
    kw = dict(image_width=spec.width, image_height=spec.height, fov=spec.fov, max_bounces=spec.max_bounces,
              background_colour=spec.background, point_light_sources=spec.point_lights, reward_mode="adaptive", seed=3)
    n = 512
    ve, vt = RayTracerVecEnv(spec.spheres, n, **kw), RayTracerVecEnv(spec.spheres, n, as_torch=True, **kw)
    assert ve.num_envs == n and ve.observation_space.shape == (18,) and ve.action_space.shape == (2,)
    o1, o2 = ve.reset(), vt.reset()
    assert o1.shape == (n, 18) and o1.dtype == np.float32 and np.array_equal(o1, o2.cpu().numpy())
    rs = np.random.RandomState(0)
    finished = 0
    for t in range(12):
        a = rs.uniform((0, 0), (np.pi / 2, 2 * np.pi), (n, 2)).astype(np.float32)
        obs, rew, dones, infos = ve.step(a)
        tobs, trew, tdones, tinfos = vt.step(torch.as_tensor(a, device="cuda"))
        assert obs.shape == (n, 18) and rew.shape == (n,) and rew.dtype == np.float32 and dones.dtype == bool and len(infos) == n
        assert np.array_equal(obs, tobs.cpu().numpy()) and np.array_equal(dones, tdones.cpu().numpy())
        np.testing.assert_allclose(rew, trew.cpu().numpy(), rtol=1e-6)
        for i in np.nonzero(dones)[0][:8]:
            assert infos[i]["terminal_observation"].shape == (18,) and "TimeLimit.truncated" in infos[i]
            assert infos[i]["reason"] in ("ray_missed", "ray_escaped", "max_bounces")
            # what SB3's logger reads from Monitor-style infos, and its DummyVecEnv rule for TimeLimit.truncated
            # (truncated and not terminated: the reference env ends max_bounces episodes with BOTH flags set)
            ep = infos[i]["episode"]
            assert set(ep) == {"r", "l", "t"} and 1 <= ep["l"] <= spec.max_bounces + 1 and ep["t"] >= 0
            assert infos[i]["TimeLimit.truncated"] is False
            assert int(tinfos["episode_length"][i]) == ep["l"] and not bool(tinfos["TimeLimit.truncated"][i])
            assert np.array_equal(infos[i]["terminal_observation"], tinfos["terminal_observation"][i].cpu().numpy())
        assert all(not infos[i] for i in np.nonzero(~dones)[0][:8])
        finished += int(dones.sum())
    assert finished > n                      # every env finished at least once and kept going: auto-reset works
    ve.close(); vt.close()
    # the scalar drop-in of the adaptive env shares the kernel: one episode, rewards as the batched env gives them
    env = AdaptiveRewardRayTracerEnv(spheres=spec.spheres, image_width=spec.width, image_height=spec.height, fov=spec.fov,
                                     max_bounces=spec.max_bounces, point_light_sources=spec.point_lights)
    assert env.light_ids == [99, 100]
    obs, info = env.reset(options={"pixel": (160, 140)})
    o, r, term, trunc, info = env.step(np.array([0.3, 1.0], np.float32))
    assert o.shape == (18,) and isinstance(r, float) and "total_reward" in info
    env.close()


def test_vec_env_adapter_under_sb3(rt):
    """The adapter is a real stable_baselines3 VecEnv when SB3 is installed: PPO.learn runs a few updates on it."""
    sb3 = pytest.importorskip("stable_baselines3")
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.ray_tracer_env import RayTracerVecEnv
    spec = scenes.build_optimized_env_scene()
    ve = RayTracerVecEnv(spec.spheres, 64, image_width=spec.width, image_height=spec.height, fov=spec.fov,
                         max_bounces=spec.max_bounces, point_light_sources=spec.point_lights, seed=1)
    assert hasattr(ve, "reset_infos") and len(ve.reset_infos) == 64
    model = sb3.PPO("MlpPolicy", ve, n_steps=16, batch_size=256, verbose=0, device="cpu")
    model.learn(total_timesteps=64 * 16 * 2)
    ve.close()


def test_env_descriptor_is_reread_on_reset(rt):
    """The reference re-reads camera / fov / max_bounces at every reset: editing them between resets takes effect."""
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.ray_tracer_env import BatchedRayTracerEnv
    spec = scenes.build_optimized_env_scene()
    kw = dict(image_width=spec.width, image_height=spec.height, max_bounces=spec.max_bounces,
              point_light_sources=spec.point_lights, precision="float64")
    pix = np.array([[160, 120], [10, 200], [300, 30], [200, 150]], np.int32)
    a = BatchedRayTracerEnv(spec.spheres, 4, fov=80, **kw)
    o80 = a.reset(options={"pixels": pix})[0].clone()
    a.fov = 50
    o50 = a.reset(options={"pixels": pix})[0].clone()
    b = BatchedRayTracerEnv(spec.spheres, 4, fov=50, **kw)
    assert np.array_equal(o50.cpu().numpy(), b.reset(options={"pixels": pix})[0].cpu().numpy())
    assert not np.array_equal(o80.cpu().numpy(), o50.cpu().numpy())
    with pytest.raises(ValueError):
        BatchedRayTracerEnv(spec.spheres, 4, precision="float16")
    a.close(); b.close()


@pytest.mark.parametrize("precision,flavour", [("f64", "rl"), ("f32", "rl"), ("f32", "fb")])
def test_step_auto_equals_step_plus_masked_reset(rt, precision, flavour):
    """rt_env_step_auto (step + restart of finished episodes in ONE launch) against the two-launch protocol it replaces:
    rt_env_step, then rt_env_reset(mask = done, pixels = the ones the fused launch drew).  Same observations, rewards,
    flags, reasons and terminal observations, step after step; replayed from a CUDA graph it gives the same again."""
    import torch
    from ray_tracer_v1_b200 import scenes, flatten_scene
    from ray_tracer_v1_b200.ray_tracer_env import BatchedRayTracerEnv
    if flavour == "fb":
        spec = scenes.build_balls_in_space(as_rendered=False)
        fs = flatten_scene(spec.spheres, spec.global_lights, [], spec.background)
        kw = dict(image_width=320, image_height=240, camera_position=(0, 0, 1), fov=60, max_bounces=5, flavour="fb")
        lo, hi = (-1.0, -1.0), (1.0, 1.0)
    else:
        spec = scenes.build_optimized_env_scene()
        fs = flatten_scene(spec.spheres, spec.global_lights, spec.point_lights, spec.background)
        kw = dict(image_width=320, image_height=240, camera_position=(0, 0, 0), fov=80, max_bounces=6, flavour="rl")
        lo, hi = (0.0, 0.0), (np.pi / 2, 2 * np.pi)
    B, T = 5000, 14                                  # not a multiple of the CTA size: ragged last block of rows
    rs = np.random.RandomState(2)
    acts = rs.uniform(lo, hi, (T, B, 2)).astype(np.float32)
    fused = BatchedRayTracerEnv(fs, B, precision=precision, seed=9, **kw)
    graph = BatchedRayTracerEnv(fs, B, precision=precision, seed=9, **kw)
    plain = BatchedRayTracerEnv(fs, B, precision=precision, seed=9, **kw)
    o0 = fused.reset(seed=9)[0].clone()
    graph.reset(seed=9)
    plain.reset(options={"pixels": fused.pixels.clone()})
    assert torch.equal(o0, plain.obs) and torch.equal(o0, graph.obs)
    finished = 0
    # FP64 (-fmad=false): bit-identical.  FP32: the restart code is inlined into two different kernels and the compiler
    # contracts it differently, so first observations of restarted episodes agree to rounding -- rewards to 1e-5, hit
    # points to 2e-4 (the floor of the RL scene is a sphere of radius 99 centred 100 away: one ulp of the intermediate
    # distance is 1.5e-5 and the hit point carries a few of them) -- and an episode whose hit / miss decision flips on
    # that rounding is dropped from the comparison (must stay below 0.1 % of the envs)
    exact = precision == "f64"
    ok = torch.ones(B, dtype=torch.bool, device="cuda")
    for t in range(T):
        obs, rew, term, trunc, info = fused.step_auto(acts[t])
        og, rg, tg, ug, ig = graph.step_auto(acts[t], graph=True)
        assert torch.equal(obs, og) and torch.equal(rew, rg) and torch.equal(term, tg) and torch.equal(info["reason"], ig["reason"])
        po, pr, pt, pu, pi = plain.step(acts[t])
        done = pt | pu
        close = lambda a, b: (a.double() - b.double()).abs() <= 1e-5 + 1e-5 * b.double().abs()      # noqa: E731
        close_obs = lambda a, b: (a.double() - b.double()).abs() <= 2e-4 + 1e-5 * b.double().abs()  # noqa: E731
        if exact:
            assert torch.equal(term, pt) and torch.equal(trunc, pu) and torch.equal(info["reason"], pi["reason"])
            assert torch.equal(rew, pr)
            assert torch.equal(info["terminal_observation"][done], po[done])      # last observation of the old episode
        else:
            assert rew.dtype == torch.float32
            ok &= (term == pt) & (trunc == pu) & (info["reason"] == pi["reason"]) & close(rew, pr)
            ok &= ~done | close_obs(info["terminal_observation"], po).all(dim=1)
        assert bool(close(info["total_reward"][ok], pi["total_reward"][ok]).all())
        if bool(done.any()):
            plain.reset(mask=done.to(torch.uint8), options={"pixels": info["pixels"].clone()})
        if exact:
            assert torch.equal(obs, plain.obs), f"step {t}"
        else:
            ok &= close_obs(obs, plain.obs).all(dim=1)
        finished += int(done.sum())
    # measured on the B200: RL 0.24 % of the episodes part ways within 14 steps (a mirror bounce magnifies the last-bit
    # difference of the two kernels' hit points into 4e-4 on the floor, or one level of the accumulated colour), FB
    # 0.04 %; gates = 3x
    gate(f"fused vs two-launch env step, {precision} {flavour}: episodes parting ways", 1.0 - float(ok.float().mean()),
         0.0 if exact else {"rl": 7.5e-3, "fb": 1.5e-3}[flavour])
    assert finished > B                              # every env restarted at least once inside the fused launches
    fused.close(); graph.close(); plain.close()


def test_unknown_schedule_bits_are_rejected(rt):
    """rt_path_params.schedule knows bits 1 and 2 only; any other bit is an error, not a silent default render."""
    from ray_tracer_v1_b200 import _native as nat
    z, fs = load_golden("path_chandelier_48x27")
    sc = nat.DeviceScene(fs)
    for schedule in (1, 8):
        p = sc.path_params(z["cam"], 16, 16, 1, int(z["max_bounces"]), float(z["mirror_threshold"]), schedule=schedule)
        with pytest.raises(nat.NativeLibraryError, match="unknown schedule bits"):
            sc.render_path_host(p, nat.F32)
    sc.close()
