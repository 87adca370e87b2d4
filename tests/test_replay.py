"""Row f3 (SURVEY.md §8f): the device-resident replay buffer keeps the ring semantics of the reference's
rl_utils.replay_buffer.ReplayBuffer.  Compared with the reference implementation itself where HSR_REFERENCE names a
checkout of it, with its recorded outputs (tests/golden/replay.npz), and through self-contained properties everywhere."""
import importlib
import os
import sys
import types
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")
REF = os.environ.get("HSR_REFERENCE", "")   # a checkout of the reference's repository


def reference_buffer_class():
    if not REF or not Path(REF, "rl_utils", "replay_buffer.py").exists():
        pytest.skip("the reference's repository is not part of this one: set HSR_REFERENCE")
    if "gym" not in sys.modules:   # rl_utils/__init__ imports gym; only its names are needed to import the package
        gym = types.ModuleType("gym"); gym.spaces = types.ModuleType("gym.spaces")
        gym.Env = object; gym.Space = object; gym.Wrapper = object
        for n in ("Box", "Discrete", "Dict", "Tuple", "Space"):
            setattr(gym.spaces, n, type(n, (), {}))
        sys.modules["gym"] = gym; sys.modules["gym.spaces"] = gym.spaces
    sys.path.insert(0, REF)
    try:
        return importlib.import_module("rl_utils.replay_buffer").ReplayBuffer
    except Exception as e:  # noqa: BLE001
        pytest.skip(f"reference rl_utils not importable here: {e!r}")
    finally:
        sys.path.remove(REF)


def batches(rng, k):
    return [rng.normal(size=(k, 17)), rng.normal(size=(k, 2)), rng.normal(size=(k,))]


def test_matches_reference_ring_semantics():
    Ref = reference_buffer_class()
    from hsr_env_b200.replay import ReplayBuffer

    rng = np.random.default_rng(0)
    ref, mine = Ref(maxlen=50), ReplayBuffer(maxlen=50, device="cpu")
    assert mine.empty and ref.empty
    for k in (7, 20, 13, 30, 5):                      # wraps around twice
        b = batches(rng, k)
        ref.extend(b); mine.extend([torch.tensor(a) for a in b])
        assert len(ref) == len(mine) and ref.pos == mine.pos and ref.full == mine.full
        for a, t in zip(ref.array(), mine.array()):
            assert np.array_equal(a, t.numpy())
        idx = rng.integers(-len(ref), 0, size=9)
        for a, t in zip(ref[idx].values, mine[torch.tensor(idx)]):
            assert np.array_equal(a, t.numpy())
        win = np.array([np.arange(i, i + 4) for i in idx])
        for a, t in zip(ref[win].values, mine[torch.tensor(win)]):
            assert np.array_equal(a, t.numpy())
    item = [rng.normal(size=17), rng.normal(size=2), np.float64(3.5)]   # mixed lengths: the reference reads it as one item
    ref.append(item); mine.append([torch.tensor(a) for a in item])
    assert ref.pos == mine.pos
    for a, t in zip(ref[np.array([-1])].values, mine[torch.tensor([-1])]):
        assert np.array_equal(a, t.numpy())


def test_ring_properties_and_sampling():
    from hsr_env_b200.replay import ReplayBuffer

    g = torch.Generator().manual_seed(0)
    rb = ReplayBuffer(maxlen=8, device="cpu", generator=g)
    for t in range(11):
        rb.append([torch.full((3,), float(t)), torch.tensor(float(t))])
    assert len(rb) == 8 and rb.full and rb.pos == 3
    obs, r = rb.array()
    assert r.tolist() == [3., 4., 5., 6., 7., 8., 9., 10.] and torch.equal(obs[:, 0], r)   # oldest -> newest
    assert rb[-1][1].item() == 10. and rb[torch.tensor([-8])][1].item() == 3.
    obs, r = rb.sample(64)
    assert obs.shape == (64, 3) and set(r.tolist()) <= set(range(3, 11)) and len(set(r.tolist())) > 4
    obs, r = rb.sample(5, seq_len=3)
    assert obs.shape == (5, 3, 3) and r.shape == (5, 3)
    rb.extend([torch.zeros(2, 3), torch.tensor([100., 101.])])
    assert rb.array()[1].tolist() == [5., 6., 7., 8., 9., 10., 100., 101.]


@pytest.mark.gpu
def test_fed_by_the_batched_env_on_the_device():
    from hsr_env_b200.env import BatchedHSREnv
    from hsr_env_b200.replay import ReplayBuffer

    n = 64
    env = BatchedHSREnv("c2_push.hsrb", None, n_envs=n, device="cuda:0", steps_per_action=10)
    rb = ReplayBuffer(maxlen=4 * n, device="cuda:0")
    obs = env.reset()
    for t in range(6):
        act = torch.rand(n, env.nu, device="cuda:0") * 2 - 1
        nxt, reward, done, info = env.step(act)
        rb.extend([obs, act, reward, nxt, done])
        obs = nxt
    assert len(rb) == 4 * n and rb.full
    o, a, r, o2, d = rb.sample(32)
    assert o.is_cuda and o.shape == (32, env.obs_dim) and d.dtype == torch.bool
    newest = rb[-n:0]
    assert torch.equal(newest[3], obs)                 # the last batch written is the newest n items
    env.close()


def _replay_golden(device):
    """Replays tests/golden/replay.npz (outputs of the reference's own ReplayBuffer, tests/golden/make_replay_golden.py)."""
    from hsr_env_b200.replay import ReplayBuffer

    g = np.load(Path(__file__).parent / "golden" / "replay.npz")
    buf = ReplayBuffer(maxlen=64, device=device)
    for s, k in enumerate(g["sizes"]):
        buf.extend([torch.tensor(g[f"in{s}_{j}"], device=device) for j in range(3)])
        assert [buf.pos, int(buf.full), len(buf)] == g[f"pos{s}"].tolist()
        for j, t in enumerate(buf.array()):
            assert np.array_equal(t.cpu().numpy(), g[f"all{s}_{j}"])
        idx = g[f"idx{s}"]
        for j, t in enumerate(buf[torch.tensor(idx, device=device)]):
            assert np.array_equal(t.cpu().numpy(), g[f"get{s}_{j}"])
        win = np.array([np.arange(i, i + 5) for i in idx])
        for j, t in enumerate(buf[torch.tensor(win, device=device)]):
            assert np.array_equal(t.cpu().numpy(), g[f"win{s}_{j}"])


def test_golden_outputs_of_the_reference_buffer_cpu():
    _replay_golden("cpu")


@pytest.mark.gpu
def test_golden_outputs_of_the_reference_buffer_on_the_device():
    _replay_golden("cuda:0")
