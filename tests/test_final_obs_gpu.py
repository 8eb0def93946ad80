"""Final observations of auto-reset worlds on the GPU.

An auto-resetting environment with final outputs (A) is stepped in lockstep with an ``auto_reset = 0`` twin (B) whose
ended worlds are reset by a masked ``reset`` after every step, and with an auto-resetting environment without final
outputs (C).  Every step: A's final record / ``obs_f32`` / ``state_f32`` / ``critic_f32`` equal B's outputs bit for bit
on the worlds that ended, and are untouched on the others; after B's reset, A's state and observations equal B's; and
A's state, records and learner layouts equal C's (asking for final outputs changes nothing else).  The same holds for a
mixed-map environment, under graph capture, for ``BatchedCopsThievesEnv``'s infos, and the learner's time-limit
bootstrap adds exactly ``gamma * V(s_final)`` to truncated transitions."""
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import load_named_map
from as_cops_and_thieves_b200.worlds import CatWorlds

pytestmark = pytest.mark.gpu

FLAT = ("obs_f32", "state_f32", "critic_f32")


def _bits(t):
    return t.contiguous().view(torch.int32)


def _final_snapshot(env):
    return [env._final_out.clone()] + [getattr(env, "final_" + n).clone() for n in FLAT]


def _check_final(A, B, before, done, what):
    """A's final outputs equal B's step outputs where `done`, and are what they were before the step elsewhere."""
    N = A.n_worlds
    rec_a, rec_b, rec_0 = A._final_out.view(N, -1), B._out.view(N, -1), before[0].view(N, -1)
    assert torch.equal(rec_a[done], rec_b[done]), f"{what}: final record"
    assert torch.equal(rec_a[~done], rec_0[~done]), f"{what}: final record of a world that did not end"
    for name, old in zip(FLAT, before[1:]):
        fa, fb = getattr(A, "final_" + name), getattr(B, name)
        if name == "obs_f32":
            fa, fb, old = fa.transpose(0, 1), fb.transpose(0, 1), old.transpose(0, 1)
        assert torch.equal(_bits(fa[done]), _bits(fb[done])), f"{what}: final {name}"
        assert torch.equal(_bits(fa[~done]), _bits(old[~done])), f"{what}: final {name} of a world that did not end"


def _check_same(A, C, what):
    assert torch.equal(A.state, C.state), f"{what}: state"
    assert torch.equal(A._out, C._out), f"{what}: records"
    for name in FLAT:
        assert torch.equal(_bits(getattr(A, name)), _bits(getattr(C, name))), f"{what}: {name}"


def _twin_run(cuda_device, cmaps, counts, steps=210, seed=5, gid0=11, **kw):
    kw = dict(device=cuda_device, gid0=gid0, seed=seed, want_critic=True, max_step_count=40, **kw)
    A = CatWorlds(cmaps, counts, auto_reset=1, want_final=True, **kw)
    B = CatWorlds(cmaps, counts, auto_reset=0, **kw)
    C = CatWorlds(cmaps, counts, auto_reset=1, **kw)
    N = A.n_worlds
    for e in (A, B, C):
        e.reset()
    g = torch.Generator().manual_seed(7)
    timeouts = captures = 0
    for t in range(steps):
        a = torch.randint(0, 4, (N, A.A), dtype=torch.uint8, generator=g).to(cuda_device)
        before = _final_snapshot(A)
        for e in (A, B, C):
            e.step(a)
        done = B.terminated.bool()
        assert torch.equal(A.terminated, B.terminated) and torch.equal(A.truncated, B.truncated), f"step {t}: flags"
        assert torch.equal(_bits(A.reward), _bits(B.reward)) and torch.equal(A.winner, B.winner), f"step {t}: rewards"
        _check_final(A, B, before, done, f"step {t}")
        _check_same(A, C, f"step {t}")
        trunc = B.truncated.bool()          # (read before the reset, which rewrites the flags of the worlds it resets)
        timeouts += int(trunc.sum())
        captures += int((done & ~trunc).sum())
        B.reset(mask=done)
        assert torch.equal(A.state, B.state), f"step {t}: state after the twin's reset"
        for name in ("obs_dist", "obs_type"):
            assert torch.equal(getattr(A, name), getattr(B, name)), f"step {t}: {name}"
        for name in FLAT:
            assert torch.equal(_bits(getattr(A, name)), _bits(getattr(B, name))), f"step {t}: {name}"
    assert timeouts > 0 and captures > 0, f"both kinds of ending must occur: {timeouts} timeouts, {captures} captures"
    assert A.overflow_counts() == (0, 0)
    for e in (A, B, C):
        e.close()


SHAPES = {"one_wave": 4096, "persistent": 12000}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kernel", ["shipped", "generic", "raster"])
@pytest.mark.parametrize("name", ["squarinth", "agh-map"])
def test_final_outputs_equal_auto_reset_0_twin(cuda_device, monkeypatch, name, kernel, shape):
    kw = {}
    if kernel == "generic":
        monkeypatch.setenv("CAT_GENERIC_KERNEL", "1")
    if kernel == "raster":
        kw["ray_list_cell"] = -1.0
    cmap = pu.named_cmap(name, free_spawn=True)
    _twin_run(cuda_device, cmap, SHAPES[shape], **kw)


def test_final_outputs_mixed_maps(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    _twin_run(cuda_device, cmaps, (1, 37, 4096))


def test_record_only_step_with_final_record(cuda_device):
    """A step that asks for the record only runs the record-only kernel; adding a final record moves it to the full
    kernel.  The two environments stay bit-identical, and the final record matches the twin's."""
    cmap = pu.named_cmap("agh-map", free_spawn=True)
    kw = dict(device=cuda_device, seed=3, want_f32=False, want_shared=False, max_step_count=40)
    A = CatWorlds(cmap, 4096, want_final=True, **kw)
    B = CatWorlds(cmap, 4096, auto_reset=0, **kw)
    C = CatWorlds(cmap, 4096, **kw)
    assert A.final_obs_f32 is None and A.final_state_f32 is None and A.final_critic_f32 is None
    N = A.n_worlds
    for e in (A, B, C):
        e.reset()
    g = torch.Generator().manual_seed(2)
    ended = 0
    for t in range(120):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
        before = A._final_out.clone().view(N, -1)
        for e in (A, B, C):
            e.step(a)
        done = B.terminated.bool()
        assert torch.equal(A._final_out.view(N, -1)[done], B._out.view(N, -1)[done]), t
        assert torch.equal(A._final_out.view(N, -1)[~done], before[~done]), t
        assert torch.equal(A.state, C.state) and torch.equal(A._out, C._out), t
        B.reset(mask=done)
        assert torch.equal(A.state, B.state), t
        ended += int(done.sum())
    assert ended > 0
    for e in (A, B, C):
        e.close()


def test_final_record_is_validated_and_ignored_by_reset_and_observe(cuda_device):
    import ctypes as C
    env = CatWorlds(pu.named_cmap("squarinth"), 64, device=cuda_device, want_critic=True, want_final=True, max_step_count=40)
    before = _final_snapshot(env)
    env.reset()
    env.observe()        # reset / observe launches get the same CatStepIO and write no final output
    for b, a in zip(before, _final_snapshot(env)):
        assert torch.equal(b, a)
    io = env._io
    acts = torch.zeros((64, 3), dtype=torch.uint8, device=cuda_device)
    io.actions, io.actions_kind = acts.data_ptr(), 0
    for bad in (dict(final_record_world_stride=env.record_bytes + 8), dict(final_record_world_stride=16),
                dict(final_record=env._final_out.data_ptr() + 4)):
        saved = {k: getattr(io, k) for k in bad}
        for k, v in bad.items():
            setattr(io, k, v)
        rc = env.L.cat_env_step(env._h, env.state.data_ptr(), C.byref(io), env._stream())
        for k, v in saved.items():
            setattr(io, k, v)
        assert rc == -1, bad
        assert b"final_record" in env.L.cat_last_error()
    env.close()


def test_graph_captured_step_with_final_outputs_equals_eager(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    env = CatWorlds(cmaps, (1, 37, 4096), device=cuda_device, seed=2, want_critic=True, want_final=True, max_step_count=40)
    N = env.n_worlds
    env.reset()
    g = torch.Generator().manual_seed(1)
    acts = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
    for _ in range(5):
        env.step(acts)
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        env.step(acts)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        env.step(acts)
    outs = lambda: [env.state, env._out, env.obs_f32, env.critic_f32] + _final_snapshot(env)  # noqa: E731
    ended = 0
    for t in range(60):
        acts.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g))
        s0 = [o.clone() for o in outs()]
        graph.replay()
        torch.cuda.synchronize()
        replay = [o.clone() for o in outs()]
        for o, v in zip(outs(), s0):
            o.copy_(v)
        env.step(acts)
        torch.cuda.synchronize()
        for r, e in zip(replay, outs()):
            assert torch.equal(_bits(r) if r.dtype == torch.float32 else r, _bits(e) if e.dtype == torch.float32 else e), t
        ended += int(env.terminated.sum())
    assert ended > 0
    env.close()


def test_batched_env_final_observation_infos(cuda_device):
    m = load_named_map("agh-map")
    env = BatchedCopsThievesEnv(m, 2048, device=cuda_device, seed=4, max_step_count=30, final_observations=True)
    w = env.worlds
    twin = CatWorlds(w.cmaps[0], 2048, device=cuda_device, want_critic=True, **{**w.params, "auto_reset": 0})
    plain = BatchedCopsThievesEnv(m, 2048, device=cuda_device, seed=4, max_step_count=30)
    assert "final_observation" not in plain.step(torch.zeros((2048, 3), dtype=torch.uint8, device=cuda_device))[4]["cop_0"]
    assert plain.final_state() is None and plain.final_critic() is None
    plain.close()
    env.reset()
    twin.reset()
    g = torch.Generator().manual_seed(8)
    first, truncs = None, 0
    for t in range(70):
        acts = {a: torch.randint(0, 4, (2048,), generator=g).to(cuda_device) for a in env.possible_agents}
        out = env.step(acts)
        twin.step(list(acts.values()))
        if first is None:
            first = out
        assert all(x is y for x, y in zip(out, first)), "a step returns the same dict objects"
        obs, rew, term, trunc, infos = out
        done = term["cop_0"].view(-1)
        assert torch.equal(done, twin.terminated.bool())
        for i, a in enumerate(env.possible_agents):
            fo = infos[a]["final_observation"]
            assert fo.shape == (2048, 2 * w.R) and fo.data_ptr() == w.final_obs_f32[i].data_ptr()
            assert torch.equal(_bits(fo[done]), _bits(twin.obs_f32[i][done])), (t, a)
        assert torch.equal(_bits(env.final_state()[done]), _bits(twin.state_f32[done]))
        assert torch.equal(_bits(env.final_critic()[done]), _bits(twin.critic_f32[done]))
        truncs += int(trunc["cop_0"].sum())
        twin.reset(mask=done)
        assert torch.equal(_bits(obs["cop_0"]), _bits(twin.obs_f32[0]))
    assert truncs > 0
    env.close()
    twin.close()


def _learner_pair(cuda_device, model, cuda_graph=False):
    m = load_named_map("squarinth")
    out = []
    for boot in (False, True):
        env = BatchedCopsThievesEnv(m, 256, device=cuda_device, seed=6, max_step_count=20, final_observations=boot)
        cfg = MAPPOConfig(rollouts=32, model=model, random_timesteps=0, learning_starts=0, cuda_graph=cuda_graph,
                          opponent_freeze_duration=0, policy_freeze_duration=0, time_limit_bootstrap=boot)
        out.append(MAPPOLearner(env, cfg, seed=0))
    return out


@pytest.mark.parametrize("model", ["lstm", "mlp"])
def test_time_limit_bootstrap_adds_gamma_v_final(cuda_device, model):
    off, on = _learner_pair(cuda_device, model)
    env = on.env
    seen = []
    step = env.step

    def recording_step(acts):
        r = step(acts)
        seen.append((on._final_value_input().clone(), r[3]["cop_0"].view(-1).clone(),
                     {a: None if on._hc[a]["value"] is None else tuple(h.clone() for h in on._hc[a]["value"])
                      for a in on.agents}))
        return r
    env.step = recording_step
    for lrn in (off, on):
        torch.manual_seed(123)
        lrn.collect()
    gamma = on.cfg.discount_factor
    n_trunc = 0
    for t, (final, trunc, hc) in enumerate(seen):
        for a in on.agents:
            r_off, r_on = off.mem[a]["rew"][t], on.mem[a]["rew"][t]
            assert torch.equal(r_on[~trunc], r_off[~trunc]), (t, a)
            with torch.no_grad():
                v, _ = on.models[a]["value"](final.unsqueeze(1), hc[a], torch.zeros((256, 1), dtype=torch.bool, device=cuda_device))
            want = torch.addcmul(r_off, v.view(-1), trunc.float(), value=gamma)
            assert torch.allclose(r_on[trunc], want[trunc], rtol=1e-6, atol=1e-6), (t, a)
            assert torch.equal(on.mem[a]["val"][t], off.mem[a]["val"][t])
        n_trunc += int(trunc.sum())
    assert n_trunc > 0
    assert torch.equal(on.mem_done, off.mem_done)


def test_time_limit_bootstrap_needs_final_observations(cuda_device):
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 32, device=cuda_device)
    with pytest.raises(ValueError, match="final observations"):
        MAPPOLearner(env, MAPPOConfig(rollouts=16, time_limit_bootstrap=True))
    env.close()


def test_time_limit_bootstrap_graph_replay_equals_eager(cuda_device):
    """With a policy whose action does not depend on the random draw, two graph-replayed rollouts equal two eager ones."""
    eager = _learner_pair(cuda_device, "lstm", cuda_graph=False)[1]
    graph = _learner_pair(cuda_device, "lstm", cuda_graph=True)[1]
    for lrn in (eager, graph):
        for a in lrn.agents:
            with torch.no_grad():
                lrn.models[a]["policy"].policy_head[-1].bias[0] += 1e4
    for it in range(3):
        for lrn in (eager, graph):
            lrn.collect()
        for a in eager.agents:
            for k in ("rew", "val", "act"):
                assert torch.equal(eager.mem[a][k], graph.mem[a][k]), (it, a, k)
        assert torch.equal(eager.mem_done, graph.mem_done)
    assert bool(eager.mem_done.any())
