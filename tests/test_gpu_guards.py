"""GPU (-m gpu): no kernel writes outside the buffers it is handed. compute-sanitizer is closed on this pool, so every output
of the step / reset / rollout / half-step paths is carved out of a larger tensor with sentinel bytes on both sides, for ragged
batch sizes (last chunk partly empty), every launch form and both observation dtypes; the packed state's slack is watched too."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GUARD = 4096
SENT = 0x5A


def guarded(torch, shape, dtype):
    n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    pad = (-n) % 16
    raw = torch.full((GUARD + n + pad + GUARD,), SENT, dtype=torch.uint8, device="cuda")
    view = raw[GUARD:GUARD + n].view(dtype).view(shape)
    return raw, view, n


def intact(raw, n):
    a = raw.cpu().numpy()
    return bool((a[:GUARD] == SENT).all() and (a[GUARD + n:] == SENT).all())


@pytest.mark.parametrize("form", [1, 4])
@pytest.mark.parametrize("f32", [False, True])
def test_outputs_stay_inside_their_buffers(form, f32):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    from hex_gym_env_b200 import HexBatch
    od = torch.float32 if f32 else torch.int8
    for N, G in ((3, 1), (5, 31), (7, 33), (11, 97), (6, 129), (19, 40)):
        C = N * N
        for variant in (0, 1):
            b = HexBatch(N, G, variant=variant, device=0, seed=N + G, agent_mode=2 if variant else 0, obs_dtype=od)
            b.set_launch_form(form)
            slack = b._state[(b._state_ptr - b._state.data_ptr()) + b.state_bytes:]
            slack.fill_(SENT)
            bufs = {k: guarded(torch, s, d) for k, (s, d) in dict(
                obs=((G, N, N), od), mask=((G, C), torch.uint8), reward=((G,), torch.float32), done=((G,), torch.uint8),
                term=((G, N, N), od), acts=((G,), torch.int32)).items()}
            b.reset(obs=bufs["obs"][1], mask=bufs["mask"][1])
            for t in range(C // 2 + 4):
                b.step(obs=bufs["obs"][1], mask=bufs["mask"][1], reward=bufs["reward"][1], done=bufs["done"][1],
                       term_obs=bufs["term"][1], actions_out=bufs["acts"][1])
            T = 5
            rb = {k: guarded(torch, (T,) + s, d) for k, (s, d) in dict(
                obs=((G, N, N), od), mask=((G, C), torch.uint8), reward=((G,), torch.float32), done=((G,), torch.uint8),
                term=((G, N, N), od), acts=((G,), torch.int32)).items()}
            b.rollout(T, obs=rb["obs"][1], mask=rb["mask"][1], reward=rb["reward"][1], done=rb["done"][1], term_obs=rb["term"][1],
                      actions_out=rb["acts"][1])
            b.encode(0, obs=bufs["obs"][1], mask=bufs["mask"][1])
            b.encode(1, obs=bufs["obs"][1], mask=bufs["mask"][1])
            torch.cuda.synchronize()
            for k, (raw, _, n) in list(bufs.items()) + list(rb.items()):
                assert intact(raw, n), (N, G, variant, form, f32, k)
            assert bool((slack == SENT).all()), (N, G, variant, form, "state slack")
            b.close()


def test_half_step_and_import_outputs_stay_inside():
    import torch
    from hex_gym_env_b200 import HexBatch
    for N, G in ((4, 33), (7, 97)):
        b = HexBatch(N, G, variant=1, device=0, seed=1, agent_mode=2, manual_opponent=True, pool_size=4)
        slack = b._state[(b._state_ptr - b._state.data_ptr()) + b.state_bytes:]
        slack.fill_(SENT)
        rew, done, term = guarded(torch, (G,), torch.float32), guarded(torch, (G,), torch.uint8), guarded(torch, (G, N, N), torch.int8)
        b.reset()
        b.opponent_catch_up()
        gen = torch.Generator(device="cuda"); gen.manual_seed(0)
        for t in range(N * N):
            a = b.sample_actions(torch.rand(G, dtype=torch.float64, device="cuda", generator=gen))
            b.half_step(0, a, reward=rew[1], done=done[1], term_obs=term[1])
            b.half_step(1, None, reward=rew[1], done=done[1], term_obs=term[1])
            b.half_step(1, None, reward=rew[1], done=done[1], term_obs=term[1])
        boards = torch.full((G, N, N), 2, dtype=torch.int8, device="cuda")
        boards[:, 0, 0] = 0; boards[:, 1, 1] = 1
        b.import_boards(boards)
        e = b.export_state()
        b.import_labels(boards, e["regions"].to(torch.uint8))
        torch.cuda.synchronize()
        for raw, _, n in (rew, done, term):
            assert intact(raw, n)
        assert bool((slack == SENT).all())
        b.close()
