"""GPU (-m gpu): every launch form of the step kernel gives the same bits. hexb_set_launch_form forces 1 / 4 warps per
32-game chunk (the cooperative sub-wave form of csrc/hexb_step.cuh); each is run against the oracle on the same seeded inputs
for every board size, for both env variants, with and without auto-reset, for single steps and hexb_rollout. Also here: float32
observations (hexb_config.obs_dtype) against the int8 ones."""
import numpy as np
import pytest

import parity
from oracle import hexref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def adapter():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import gpu_adapter
    return gpu_adapter


@pytest.mark.parametrize("N", list(range(3, 20)))
@pytest.mark.parametrize("form", [4])
def test_every_board_size_every_form(adapter, N, form):
    """SelfPlayEnv, fused random agent, random agent colour, auto-reset: long enough that games finish, restart and the opponent
    opens; G is ragged (last chunk partly empty)."""
    G = 330 if N <= 11 else 150
    T = N * N // 2 + 12
    parity.versus_oracle(adapter.make_with(launch_form=form), hexref.KIND_SELFPLAY_B, N, G, T, seed=100 * form + N, fused=True,
                         agent_mode=2, check_state_every=5)


@pytest.mark.parametrize("form", [1, 4])
@pytest.mark.parametrize("N", [4, 5, 7, 11])
def test_forms_external_actions_illegal_moves(adapter, form, N):
    parity.versus_oracle(adapter.make_with(launch_form=form), hexref.KIND_SELFPLAY_B, N, 500, N * N, seed=7 + N, fused=False,
                         agent_mode=1, illegal_rate=0.08, check_state_every=4)


@pytest.mark.parametrize("form", [4])
@pytest.mark.parametrize("kind", [hexref.KIND_SELFPLAY_B, hexref.KIND_ENV_A])
def test_forms_no_auto_reset(adapter, form, kind):
    """Without auto-reset the opponent-view rows (games the agent's own ply finished) are rewritten after the chunk encode."""
    kw = dict(agent_mode=2) if kind == hexref.KIND_SELFPLAY_B else {}
    for N in (4, 5):
        parity.versus_oracle(adapter.make_with(launch_form=form), kind, N, 500, 30, seed=3, fused=False, auto_reset=False,
                             illegal_rate=0.1, **kw)


@pytest.mark.parametrize("form", [4])
@pytest.mark.parametrize("N", [3, 7, 10])
def test_forms_variant_a(adapter, form, N):
    parity.versus_oracle(adapter.make_with(launch_form=form), hexref.KIND_ENV_A, N, 700, N * N, seed=5 + N, fused=True,
                         check_state_every=3)


@pytest.mark.parametrize("form", [1, 4])
@pytest.mark.parametrize("N", [5, 6, 11])
def test_forms_rollout_equals_steps(adapter, form, N):
    parity.rollout_equals_steps(adapter.make_with(launch_form=form), hexref.KIND_SELFPLAY_B, N, 200, 20, seed=form + N, agent_mode=2)


@pytest.mark.parametrize("form", [4])
def test_forms_api_fuzz(adapter, form):
    for seed in range(6):
        parity.api_fuzz(adapter.make_with(launch_form=form), 50 * form + seed, T=40)


def test_forms_1_and_4_same_trajectory_large_batch(adapter):
    """20,000 games of 7x7 and 11x11: the two forms against each other (obs, mask, reward, done, actions, state, statistics);
    no other form is accepted."""
    import torch
    from hex_gym_env_b200 import HexBatch, HexbError
    for N, G, T in ((7, 20000, 45), (11, 20000, 70)):
        envs = []
        for form in (1, 4):
            b = HexBatch(N, G, variant=1, device=0, seed=5, agent_mode=2)
            b.set_launch_form(form)
            b.reset()
            envs.append(b)
        for form in (2, 8):
            with pytest.raises(HexbError):
                envs[0].set_launch_form(form)
        for t in range(T):
            outs = [b.step(want_actions=True, want_term=True) for b in envs]
            for o in outs[1:]:
                for k in ("obs", "mask", "reward", "done", "actions"):
                    assert torch.equal(o[k], outs[0][k]), (N, t, k)
                d = outs[0]["done"].bool()
                assert torch.equal(o["term_obs"][d], outs[0]["term_obs"][d]), (N, t, "term_obs")
        ref = envs[0].export_state()
        for b in envs[1:]:
            e = b.export_state()
            for k in ref:
                assert torch.equal(e[k], ref[k]), (N, k)
            assert torch.equal(b.stats(), envs[0].stats())


# ------------------------------------------------------------------------------------------------ float32 observations
@pytest.mark.parametrize("form", [1, 4])
@pytest.mark.parametrize("N", [3, 5, 6, 11, 14])
def test_f32_observations_selfplay(adapter, form, N):
    parity.versus_oracle(adapter.make_with(launch_form=form, obs_f32=True), hexref.KIND_SELFPLAY_B, N, 333, N * N // 2 + 10, seed=N,
                         fused=True, agent_mode=2, check_state_every=6)


def test_f32_observations_variant_a_and_no_auto_reset(adapter):
    parity.versus_oracle(adapter.make_with(obs_f32=True), hexref.KIND_ENV_A, 7, 400, 49, seed=1, fused=True)
    parity.versus_oracle(adapter.make_with(obs_f32=True), hexref.KIND_SELFPLAY_B, 5, 400, 30, seed=2, fused=False, auto_reset=False,
                         illegal_rate=0.1, agent_mode=2)


def test_f32_rollout_and_half_steps(adapter):
    parity.rollout_equals_steps(adapter.make_with(obs_f32=True), hexref.KIND_SELFPLAY_B, 6, 200, 16, seed=4, agent_mode=2)
    parity.golden_oppmodel(adapter.make_with(obs_f32=True), "oppmodel_N7_a2.npz")
    parity.sample_board_flow(adapter.make_with(obs_f32=True), 5, 100, 20)


def test_f32_dtype_is_enforced(adapter):
    import torch
    from hex_gym_env_b200 import HexBatch
    b = HexBatch(5, 64, variant=1, device=0, obs_dtype=torch.float32)
    obs, mask = b.reset()
    assert obs.dtype == torch.float32 and mask.dtype == torch.uint8
    with pytest.raises(ValueError):
        b.step(obs=torch.empty((64, 5, 5), dtype=torch.int8, device="cuda"))
    o = b.step(want_term=True)
    assert o["obs"].dtype == torch.float32 and o["term_obs"].dtype == torch.float32
    assert set(np.unique(o["obs"].cpu().numpy()).tolist()) <= {-1.0, 0.0, 1.0}
    with pytest.raises(ValueError):
        HexBatch(5, 64, variant=1, device=0, obs_dtype=torch.float16)
