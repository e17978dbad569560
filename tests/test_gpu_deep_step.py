"""GPU (-m gpu): the deep form of the env step - one warp per 32-game chunk with the one-row-per-pass relabel sweep
(hexb_step_kernel<N, KIND, BATCHED=false>, csrc/hexb_step.cuh) - at every board size and in every regime its launcher picks.

launch_tile chooses the kernel from the batch size alone. With S SMs, one wave holds 32*S chunk-warps, and a batch of G games
is Gpad = ceil(G/128)*128 games, chunks = Gpad/32:
  chunks <= S                        the cooperative form, hexb_coop_kernel (pinned against the oracle in test_gpu_forms.py)
  chunks <= S*28 (N <= 8), S*12      the warp form with the several-rows sweep (BATCHED=true), Params::early = 1
  above that, chunks <= S*32         R1: the one-row sweep, early = 1 (record half of the step before the chunk has landed)
  chunks > S*32                      R2: the one-row sweep, early = 0 (records read after the bulk copy)
  packed state > 64 MiB              R3: as R2, plus the L2 eviction hints of the first keep_chunks chunks, and compressible memory
                                     by default
Small batches never reach R1-R3, so these tests use batch sizes derived from the device's SM count (regimes() below, e.g.
141,933 / 154,957 / 168,997 games of 19x19 at 148 SMs) and check that the launch really runs the kernel they mean to test.

Every run is compared three ways: byte for byte against a twin handle forced to the cooperative form (same seed, same actions),
against the oracle on windows of the global game index (first chunk, chunk boundaries, the first/second wave boundary, the
keep_chunks boundary, the ragged last chunk), and against size-independent properties over all games (tests/properties.py).
"""
import ctypes
import gc
import math
import re

import numpy as np
import pytest
import torch

import properties
from oracle import hexref
from parity import eq
from test_gpu_fullsize import _windows

pytestmark = pytest.mark.gpu

HINT_MIN_BYTES = 64 << 20    # hexb_create: the L2 hints are used when the packed state is larger than this...
KEEP_BYTES = 20 << 20        # ...and keep this much of it (keep_chunks whole chunks) in L2 from one step to the next
REGIMES = ("R1", "R2", "R3")
DEV = "cuda"
OUT_KEYS = ("obs", "mask", "reward", "done", "actions")
STATE_KEYS = ("board", "regions", "region_counter", "cur", "done", "winner", "agent")


@pytest.fixture(autouse=True)
def _free_device_memory():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _state_bytes(N, G):
    from hex_gym_env_b200 import _native
    cfg = _native.HexbConfig(board_size=N, variant=1, num_games=G, agent_mode=2)
    return int(_native.lib().hexb_state_bytes(ctypes.byref(cfg)))


def launch_of(N, G, sms):
    """What launch_tile does for a single env step of G games of NxN on a device with `sms` SMs (csrc/hexb_step.cuh), with the
    chunk size taken from the library's own hexb_state_bytes."""
    chunk_bytes = (_state_bytes(N, 512) - _state_bytes(N, 256)) // 8      # 8 more chunks of 32 games
    chunks = (G + 127) // 128 * 4
    state = chunks * chunk_bytes
    return dict(G=G, chunks=chunks, coop=chunks <= sms, small=chunks <= sms * (28 if N <= 8 else 12),
                early=chunks <= 32 * sms, keep_chunks=KEEP_BYTES // chunk_bytes if state > HINT_MIN_BYTES else 0,
                chunk_bytes=chunk_bytes)


def regimes(N, sms):
    """The batch sizes of R1, R2 and R3 at NxN, and a control batch: the largest one that still runs the several-rows sweep.
    Each size leaves its last chunk ragged and is asserted to land in the regime it names."""
    cb = launch_of(N, 128, sms)["chunk_bytes"]
    sizes = dict(R1=960 * sms - 147,                                               # ~30 chunks per SM: past the several-rows limit, inside one wave
                 R2=1048 * sms - 147,                                              # ~2 % past one wave; under 64 MiB of state even at 19x19
                 R3=int(1.05 * HINT_MIN_BYTES * 32 / cb) // 128 * 128 + 37,        # 1.05 x 64 MiB of state, two empty chunks in the last tile
                 control=32 * sms * (28 if N <= 8 else 12) - 3)
    out = {}
    for name, G in sizes.items():
        L = launch_of(N, G, sms)
        assert G % 32 != 0, (N, name, G)
        assert not L["coop"], (N, name, L)
        if name == "control":
            assert L["small"] and L["early"] and L["keep_chunks"] == 0, (N, name, L)
        else:
            assert not L["small"], (N, name, L)
            assert L["early"] == (name == "R1"), (N, name, L)
            assert (L["keep_chunks"] > 0) == (name == "R3"), (N, name, L)
        if name == "R3":
            assert L["chunks"] > L["keep_chunks"] and _state_bytes(N, G) >= HINT_MIN_BYTES, (N, L)
        out[name] = L
    return out


def windows(N, regime, sms):
    """Oracle windows (start, length) for a regime: test_gpu_fullsize's windows around the first/second wave boundary (R1 has a
    single wave: there the window sits where the several-rows limit would end the batch), plus the keep_chunks boundary in R3."""
    L = regimes(N, sms)[regime]
    edge = 32 * 32 * sms if regime != "R1" else 32 * sms * (28 if N <= 8 else 12)
    assert edge < L["G"]
    wins = _windows(L["G"], edge)
    if regime == "R3":
        wins.append((32 * L["keep_chunks"] - 16, 32))
    return wins


def steps_for(N):
    """Past the mean episode of about 0.45*N^2 env steps: games restart and long chains merge."""
    return max(24, math.ceil(0.6 * N * N))


def _bytes(t):
    return t.reshape(t.shape[0], -1).view(torch.uint8)


def _differing(got, want, keys):
    """Keys whose tensors differ in any byte (one synchronisation for all of them)."""
    flags = torch.stack([(_bytes(got[k]) != _bytes(want[k])).any() for k in keys]).tolist()
    return [k for k, f in zip(keys, flags) if f]


def same_as_twin(what, got, want, keys):
    bad = _differing(got, want, keys)
    if bad:
        g = int((_bytes(got[bad[0]]) != _bytes(want[bad[0]])).any(1).nonzero()[0])
        raise AssertionError("%s: %s differ from the cooperative form (first differing game %d)" % (what, bad, g))


def _host(t, idx, dim=0):
    """Rows `idx` of a device tensor as numpy; float32 observations hold the same small integers as the int8 ones."""
    a = t.index_select(dim, idx).cpu().numpy()
    if a.dtype == np.float32 and a.ndim >= 3:
        b = a.astype(np.int8)
        assert np.array_equal(b.astype(np.float32), a), "float32 observation with a non-integer value"
        return b
    return a


class Windows(object):
    """The oracle on windows of the global game index, stepped in lockstep with the device."""

    def __init__(self, wins, kind, N, **kw):
        self.wins = wins
        self.refs = [hexref.RefBatch(kind, N, n, game_offset=s, **kw) for s, n in wins]
        self.offs = np.cumsum([0] + [n for _, n in wins])
        self.idx = torch.cat([torch.arange(s, s + n) for s, n in wins]).to(DEV)

    def reset(self, what, obs, mask):
        ho, hm = _host(obs, self.idx), _host(mask, self.idx)
        for (s, n), o, ref in zip(self.wins, self.offs, self.refs):
            ro, rm = ref.reset()
            eq(ho[o:o + n], ro, "%s reset obs, window %d+%d" % (what, s, n))
            eq(hm[o:o + n], rm, "%s reset mask, window %d+%d" % (what, s, n))

    def step(self, what, host, actions=None, auto_reset=True):
        """host: the device's outputs of this step on the window rows (numpy); actions: the external actions of the whole batch."""
        for (s, n), o, ref in zip(self.wins, self.offs, self.refs):
            r = ref.step(None if actions is None else actions[s:s + n], auto_reset=auto_reset, want_term=True)
            w = "%s, window %d+%d: " % (what, s, n)
            for k in OUT_KEYS:
                eq(host[k][o:o + n], r[k], w + k)
            if auto_reset:        # only games that finished in this step get a terminal observation, and every row was zeroed
                eq(host["term_obs"][o:o + n], r["term_obs"], w + "term_obs")
            else:                 # without auto-reset the terminal observation is the observation itself
                d = r["done"].astype(bool)
                eq(host["obs"][o:o + n][d], r["term_obs"][d], w + "term_obs")

    def final(self, what, env):
        e = env.export_state()
        host = {k: _host(e[k], self.idx) for k in STATE_KEYS}
        for (s, n), o, ref in zip(self.wins, self.offs, self.refs):
            re_ = ref.export()
            for k in STATE_KEYS:
                eq(host[k][o:o + n], re_[k], "%s final %s, window %d+%d" % (what, k, s, n))
        return e


def check_variant_a(obs, mask, opponent_first):
    """test_config2_full_size's properties of variant-A observations (agent BLACK to move, board codes 0 / 1 / 2 = empty)."""
    G, N, _ = obs.shape
    assert torch.equal(mask.view(G, N, N) != 0, obs == 2), "mask != empty cells"
    nb, nw = (obs == 0).sum(dim=(1, 2)), (obs == 1).sum(dim=(1, 2))
    assert torch.equal(nw - nb, torch.full_like(nb, int(opponent_first))), "stone counts do not match who opened"
    assert not properties.connects(obs == 0, 0).any() and not properties.connects(obs == 1, 1).any(), "a live game is won"


def _pair(N, G, **kw):
    from hex_gym_env_b200 import HexBatch
    deep = HexBatch(N, G, device=0, **kw)
    twin = HexBatch(N, G, device=0, **kw)
    twin.set_launch_form(4)      # the cooperative form at any batch size
    return deep, twin


def _external_actions(env, mask, gen):
    """Legal actions from HexBatch.sample_actions, with about 3 % replaced by -2, -1, C, C+1 or an occupied cell."""
    G, C = env.G, env.C
    u = torch.rand(G, dtype=torch.float64, device=DEV, generator=gen)
    legal = env.sample_actions(u).to(torch.int64)
    bad = torch.rand(G, device=DEV, generator=gen) < 0.03
    pick = torch.randint(0, 5, (G, 1), device=DEV, generator=gen)
    occupied = (mask == 0).to(torch.int8).argmax(1)      # the first occupied cell (cell 0, a legal move, on an empty board)
    full = lambda v: torch.full((G,), v, dtype=torch.int64, device=DEV)   # noqa: E731
    wrong = torch.stack([full(-2), full(-1), full(C), full(C + 1), occupied], 1).gather(1, pick).squeeze(1)
    return torch.where(bad, wrong, legal).to(torch.int32)


def play(N, regime, seed, T=None, variant=1, agent_mode=2, opponent_first=False, auto_reset=True, eval_state=False,
         obs_dtype=torch.int8, external=False, compressible=None):
    """T env steps of a deep launch next to the cooperative twin and the oracle windows (see the module docstring)."""
    sms = _sms()
    L = regimes(N, sms)[regime]
    G, T = L["G"], T or steps_for(N)
    what = "N=%d %s G=%d" % (N, regime, G)
    deep, twin = _pair(N, G, variant=variant, seed=seed, agent_mode=agent_mode, opponent_first=opponent_first,
                       auto_reset=auto_reset, eval_state=eval_state, obs_dtype=obs_dtype, compressible=compressible)
    if compressible is None:
        assert deep.compressible == (regime == "R3"), (what, deep.memory_kind)
    kind = hexref.KIND_SELFPLAY_B if variant == 1 else hexref.KIND_ENV_A
    win = Windows(windows(N, regime, sms), kind, N, seed=seed, agent_mode=agent_mode if variant == 1 else 0,
                  opponent_first=opponent_first, eval_state=eval_state)
    od, md = deep.reset()
    ot, mt = twin.reset()
    same_as_twin(what + " reset", dict(obs=od, mask=md), dict(obs=ot, mask=mt), ("obs", "mask"))
    win.reset(what, od, md)
    agent = deep.export_state()["agent"] if variant == 1 else None
    term_d = torch.zeros((G, N, N), dtype=obs_dtype, device=DEV)
    term_t = torch.zeros_like(term_d)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(seed)
    mask_now = md
    every = max(1, T // 4)
    for t in range(T):
        w = "%s step %d" % (what, t)
        acts = _external_actions(deep, mask_now, gen) if external else None
        term_d.zero_()
        term_t.zero_()
        a = deep.step(acts, term_obs=term_d, want_actions=True)
        b = twin.step(acts, term_obs=term_t, want_actions=True)
        same_as_twin(w, a, b, OUT_KEYS + ("term_obs",))
        host = {k: _host(a[k], win.idx) for k in OUT_KEYS + ("term_obs",)}
        win.step(w, host, None if acts is None else acts.cpu().numpy(), auto_reset)
        mask_now = a["mask"]
        if t % every == every - 1 or t == T - 1:
            if variant == 1 and auto_reset and not external:
                properties.check_selfplay_step(a["obs"], a["mask"], a["reward"], a["done"], agent, term_d)
            elif variant == 0:
                check_variant_a(a["obs"], a["mask"], opponent_first)
    st = deep.stats()
    assert torch.equal(st, twin.stats()), (what, "stats", st.tolist(), twin.stats().tolist())
    if auto_reset:
        assert int(st[6]) == G * T, (what, "env_steps", st.tolist())
    assert torch.equal(deep.state_dict()["state"], twin.state_dict()["state"]), (what, "packed state")
    e = win.final(what, deep)
    properties.check_exported_labels(e["board"], e["regions"], 0 if variant == 1 else 2)
    deep.close()
    twin.close()


def _seed(N, regime, salt=0):
    return 1000 * N + 10 * REGIMES.index(regime) + salt


# ------------------------------------------------------------------------------------------------ 2. the kernel each launch runs
def _kernels_of(fn):
    """Template names of the hexb kernels fn() launches, as the profiler reports them."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], acc_events=True) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({m for e in prof.events() for m in re.findall(r"hexb_\w+<[^<>]*>", e.name)})


@pytest.mark.parametrize("N", list(range(3, 20)))
def test_deep_launches_run_the_one_row_kernels(N):
    """A single step and a rollout at R1, R2 and R3 run hexb_step_kernel<N, 1, false> and <N, 2, false>; the control batch, at the
    several-rows limit, runs <N, 1, true> and <N, 2, true>. If launch_tile's rule changes, this fails instead of the other tests
    here quietly checking another form."""
    from hex_gym_env_b200 import HexBatch
    for name, L in regimes(N, _sms()).items():
        b = HexBatch(N, L["G"], variant=1, device=0, seed=N, agent_mode=2)
        b.reset()
        form = "true" if name == "control" else "false"
        got = _kernels_of(lambda: b.step(want_actions=True, want_term=True))
        assert got == ["hexb_step_kernel<%d, 1, %s>" % (N, form)], (N, name, L, got)
        got = _kernels_of(lambda: b.rollout(2))
        assert got == ["hexb_step_kernel<%d, 2, %s>" % (N, form)], (N, name, L, got)
        b.close()


# ------------------------------------------------------------------------------------------------ 3. every board size, every regime
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("N", list(range(3, 20)))
def test_deep_step_every_board_size(N, regime):
    """The bench workload: SelfPlayEnv, agent colour random per game, fused agent, auto-reset, terminal observations, actions."""
    play(N, regime, _seed(N, regime))


# ------------------------------------------------------------------------------------------------ 4. options the kernel branches on
OPTIONS = {
    "agent_black": dict(agent_mode=0),
    "agent_white": dict(agent_mode=1),                              # stored transposed
    "external_actions": dict(external=True),                        # legal and illegal ones, the same for twin and oracle
    "no_auto_reset": dict(auto_reset=False),                        # finished games shown from the opponent's side
    "variant_a": dict(variant=0, agent_mode=0),
    "variant_a_opponent_first": dict(variant=0, agent_mode=0, opponent_first=True),
    "float32_obs": dict(obs_dtype=torch.float32),
    "eval_state": dict(eval_state=True),
}


@pytest.mark.parametrize("option", list(OPTIONS))
@pytest.mark.parametrize("regime", ("R1", "R2"))
@pytest.mark.parametrize("N", [3, 6, 7, 9, 12, 19])
def test_deep_step_options(N, regime, option):
    """W = 1..12 record words, odd and even rows, both sides of the N <= 8 limit of the several-rows sweep."""
    play(N, regime, _seed(N, regime, 1 + list(OPTIONS).index(option)), **OPTIONS[option])


@pytest.mark.parametrize("N", [7, 19])
def test_deep_step_l2_hints_in_ordinary_memory(N):
    """R3's L2 eviction hints without compressible memory."""
    play(N, "R3", _seed(N, "R3", 9), compressible=False)


# ------------------------------------------------------------------------------------------------ 5. deep rollouts
def roll(N, regime, seed, obs_dtype=torch.int8, T=24, launches=2):
    """`launches` back-to-back rollout(T) launches of a deep batch == T * launches single steps of the cooperative twin, byte for
    byte (outputs [T,G,...], terminal observations, packed state, statistics), and == the oracle on the windows."""
    sms = _sms()
    L = regimes(N, sms)[regime]
    G, C = L["G"], N * N
    what = "N=%d %s G=%d rollout" % (N, regime, G)
    deep, twin = _pair(N, G, variant=1, seed=seed, agent_mode=2, obs_dtype=obs_dtype)
    win = Windows(windows(N, regime, sms), hexref.KIND_SELFPLAY_B, N, seed=seed, agent_mode=2)
    od, md = deep.reset()
    ot, mt = twin.reset()
    same_as_twin(what + " reset", dict(obs=od, mask=md), dict(obs=ot, mask=mt), ("obs", "mask"))
    win.reset(what, od, md)
    agent = deep.export_state()["agent"]
    ro = dict(obs=torch.empty((T, G, N, N), dtype=obs_dtype, device=DEV), mask=torch.empty((T, G, C), dtype=torch.uint8, device=DEV),
              reward=torch.empty((T, G), dtype=torch.float32, device=DEV), done=torch.empty((T, G), dtype=torch.uint8, device=DEV),
              term_obs=torch.empty((T, G, N, N), dtype=obs_dtype, device=DEV), actions=torch.empty((T, G), dtype=torch.int32, device=DEV))
    term_t = torch.zeros((G, N, N), dtype=obs_dtype, device=DEV)
    for rep in range(launches):
        ro["term_obs"].zero_()
        deep.rollout(T, obs=ro["obs"], mask=ro["mask"], reward=ro["reward"], done=ro["done"], term_obs=ro["term_obs"],
                     actions_out=ro["actions"])
        for t in range(T):
            w = "%s launch %d step %d" % (what, rep, t)
            term_t.zero_()
            b = twin.step(term_obs=term_t, want_actions=True)
            same_as_twin(w, {k: v[t] for k, v in ro.items()}, b, OUT_KEYS + ("term_obs",))
        host = {k: _host(v, win.idx, dim=1) for k, v in ro.items()}
        for t in range(T):
            win.step("%s launch %d step %d" % (what, rep, t), {k: v[t] for k, v in host.items()})
        properties.check_selfplay_step(ro["obs"][T - 1], ro["mask"][T - 1], ro["reward"][T - 1], ro["done"][T - 1], agent,
                                       ro["term_obs"][T - 1])
    st = deep.stats()
    assert torch.equal(st, twin.stats()), (what, "stats", st.tolist(), twin.stats().tolist())
    assert int(st[6]) == G * T * launches, (what, "env_steps", st.tolist())
    assert torch.equal(deep.state_dict()["state"], twin.state_dict()["state"]), (what, "packed state")
    e = win.final(what, deep)
    properties.check_exported_labels(e["board"], e["regions"], 0)
    deep.close()
    twin.close()


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("N", list(range(3, 20)))
def test_deep_rollout_every_board_size(N, regime):
    roll(N, regime, _seed(N, regime, 5))


@pytest.mark.parametrize("N", [7, 19])
def test_deep_rollout_float32_observations(N):
    roll(N, "R3", _seed(N, "R3", 6), obs_dtype=torch.float32)
