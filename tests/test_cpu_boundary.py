"""CPU-only checks of the boundary and host logic: the C-ABI library builds, loads and exports every symbol that
include/ouzelum_b200.h declares (no compute calls -- there is no GPU here), struct mirrors agree with the C defaults,
the counter RNG passes the Random123 known-answer vectors, and the product refuses to run without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build_script():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ozl_build", os.path.join(ROOT, "ouzelum_b200", "build.py"))
    build = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(build)
    return build


@pytest.fixture(scope="module")
def lib():
    _build_script().build()            # no-op when the in-tree .so is newer than its sources
    from ouzelum_b200 import _lib
    return _lib


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "ouzelum_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ozl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    names = declared_symbols()
    assert len(names) >= 24, names
    so = ctypes.CDLL(lib.LIB_PATH)
    missing = [n for n in names if not hasattr(so, n)]
    assert not missing, f"declared in include/ouzelum_b200.h but not exported: {missing}"
    bound = set(lib._SIGS)
    assert set(names) == bound, f"ctypes binding and header disagree: {set(names) ^ bound}"
    assert lib.lib.ozl_abi_version() == lib.OZL_ABI_VERSION


def test_library_is_sm100a_only_and_uses_bulk_copy(lib):
    import subprocess
    cuobjdump = os.path.join(os.path.dirname(_build_script().NVCC), "cuobjdump")     # the toolkit that built the library, PATH or not
    out = subprocess.run([cuobjdump, "-lelf", lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs
    sass = subprocess.run([cuobjdump, "-sass", lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass                      # TMA bulk store of the observation tile (Blackwell/Hopper async copy engine)
    assert "quad_step_kernel" in sass


def test_cfg_defaults_match_reference_yaml_and_urdf(lib):
    from ouzelum_b200 import x500
    c = lib.default_cfg(4096).to_dict()
    assert c["max_episode_length"] == 2000 and c["target_period"] == 500 and c["substeps"] == 2      # Ouzelum.yaml:10,21
    assert c["dt"] == np.float32(0.01) and c["gravity_z"] == np.float32(-9.81)
    assert c["clip_actions"] == 1.0 and c["clip_obs"] == 5.0 and c["thrust_rate"] == 20.0 and c["thrust_max"] == 2000.0
    assert c["die_dist"] == 8.0 and c["die_z"] == 0.5 and c["up_coef"] == 5.0
    assert c["spawn_lo"] == tuple(np.float32([-1.5, -1.5, -0.2])) and c["spawn_range"] == tuple(np.float32([3.0, 3.0, 1.7]))
    for k in ("mass", "ixx", "iyy", "izz", "arm", "com_z", "max_angvel"):
        assert c[k] == float(np.float32(getattr(x500, k.upper()))), k
    assert abs(x500.MASS - 2.0643077) < 1e-6 and abs(x500.COM_Z - 0.0093457) < 1e-6                   # SURVEY 8a row P
    assert abs(x500.IXX - 0.029275) < 2e-6 and abs(x500.IZZ - 0.0440) < 1e-6
    with pytest.raises(KeyError):
        lib.default_cfg(8, no_such_field=1)


def test_oracle_constants_agree_with_product(lib):
    from oracle import x500 as ox
    from oracle.quad_step import default_cfg
    from ouzelum_b200 import x500
    for k in ("MASS", "COM_Z", "IXX", "IYY", "IZZ", "ARM", "MAX_ANGVEL"):
        assert abs(getattr(ox, k) - getattr(x500, k)) < 1e-15, k
    o, c = default_cfg(64), lib.default_cfg(64).to_dict()
    for k, v in c.items():
        if k in ("collect_metrics",):
            continue
        ov = o[k]
        if isinstance(v, tuple):
            assert np.array_equal(np.asarray(ov, np.float32), np.asarray(v, np.float32)), k
        elif isinstance(v, float):
            assert np.float32(ov) == np.float32(v), k
        else:
            assert ov == v, k


def test_philox_known_answers():
    from oracle.philox import philox4x32_10, u01, mulhi
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]                     # Random123 kat_vectors, philox4x32 10 rounds
    for ctr, key, want in kat:
        got = philox4x32_10(*ctr, *key)
        assert tuple(int(x) for x in got) == want
    r = np.array([0, 255, 256, 0xFFFFFFFF], dtype=np.uint32)
    assert list(u01(r)) == [0.0, 0.0, 2.0 ** -24, 1.0 - 2.0 ** -24]
    assert list(mulhi(r, 2000)) == [0, 0, 0, 1999]


def test_product_refuses_to_run_without_cuda(lib, monkeypatch):
    import torch
    import ouzelum_b200
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)       # on a machine with a GPU the product must see none
    with pytest.raises(RuntimeError, match="no CPU"):
        ouzelum_b200.make(0, "Ouzelum", 16, sim_device="cpu", rl_device="cpu")
    with pytest.raises(RuntimeError, match="no CUDA device|no CPU"):
        ouzelum_b200.make(0, "Ouzelum", 16)
    with pytest.raises(KeyError):
        ouzelum_b200.make(0, "NoSuchTask", 16)
    from ouzelum_b200.controllers import Controller, control
    with pytest.raises(RuntimeError):
        Controller(control(), "cpu")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ouzelum_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{f} imports the oracle"


def _repository_files():
    """Paths (relative to the root) of the repository's files: what git tracks in a checkout; in a copy of the tree without
    .git, every file that the patterns of .gitignore do not exclude (last matching pattern wins, `!` re-includes)."""
    import fnmatch
    import subprocess
    if os.path.isdir(os.path.join(ROOT, ".git")):
        r = subprocess.run(["git", "-C", ROOT, "ls-files", "-z"], capture_output=True, text=True, timeout=120)
        if r.returncode == 0:
            return [f for f in r.stdout.split("\0") if f]
    rules = []
    for line in open(os.path.join(ROOT, ".gitignore")).read().splitlines():
        line = line.strip()
        if line and not line.startswith("#"):
            rules.append((line.startswith("!"), line.lstrip("!")))

    def ignored(rel):
        parts, out = rel.split("/"), False
        for negate, pat in rules:
            dir_only, pat = pat.endswith("/"), pat.strip("/")
            heads = parts[:-1] if dir_only else parts              # a directory pattern matches the directories above the file
            if "/" in pat:                                         # anchored at the root
                hit = any(fnmatch.fnmatchcase("/".join(parts[:i + 1]), pat) for i in range(len(heads)))
            else:
                hit = any(fnmatch.fnmatchcase(p, pat) for p in heads)
            if hit:
                out = not negate
        return out
    files = []
    for dirpath, dirnames, filenames in os.walk(ROOT):
        dirnames[:] = [d for d in dirnames if d != ".git"]
        for f in filenames:
            rel = os.path.relpath(os.path.join(dirpath, f), ROOT).replace(os.sep, "/")
            if not ignored(rel):
                files.append(rel)
    return files


def test_every_repository_file_is_at_most_1_mb():
    """Stored test vectors are sampled or split so that no file of the repository exceeds 1 MB (10^6 bytes)."""
    files = _repository_files()
    assert "bench.py" in files and "tests/golden/rpo_lstm_actor.npz" in files and "ouzelum_b200/libouzelum_b200.so" not in files
    sizes = {f: os.path.getsize(os.path.join(ROOT, f)) for f in files if os.path.isfile(os.path.join(ROOT, f))}
    big = {f: s for f, s in sizes.items() if s > 1_000_000}
    assert not big, big


def test_task_config_mirrors_yaml():
    import ouzelum_b200
    c = ouzelum_b200.task_config("Ouzelum", 123)
    assert c["env"]["numEnvs"] == 123 and c["env"]["maxEpisodeLength"] == 2000 and c["sim"]["substeps"] == 2
    assert c["env"]["clipObservations"] == 5.0 and c["task"]["randomize"] is False
    from ouzelum_b200.spaces import Box
    b = Box(np.ones(4) * -1.0, np.ones(4) * 1.0)
    assert b.shape == (4,) and b.contains(b.sample())


def test_recurrent_actor_cell_equals_nn_lstm():
    """The GEMM-form single-step LSTM cell of the rollout policy equals nn.LSTM on the same parameters (CPU, torch only)."""
    import torch
    from ouzelum_b200.rollout import RecurrentActor
    torch.manual_seed(0)
    a = RecurrentActor()
    n = 64
    obs, done = torch.randn(n, 13), (torch.rand(n) < 0.3).float()
    st = (torch.randn(1, n, 128), torch.randn(1, n, 128))
    with torch.no_grad():
        act, logp, ent, s1 = a(obs, st, done)
        keep = (1 - done).view(1, -1, 1)
        _, s2 = a.lstm(a.network(obs).unsqueeze(0), (keep * st[0], keep * st[1]))
    assert act.shape == (n, 4) and logp.shape == (n,) and ent.shape == (n,)
    assert (s1[0] - s2[0]).abs().max() < 1e-5 and (s1[1] - s2[1]).abs().max() < 1e-5


def test_recurrent_actor_equals_reference_actor_fixture():
    """(f)1: `RecurrentActor` against the reference's UNMODIFIED `RPO-LSTM/model.py` Actor (tests/golden/rpo_lstm_actor.npz, made
    by running that module on CPU; its state dict is stored in rpo_lstm_actor_sd_{mlp,lstm}.npz): it must LOAD the reference's
    state dict (the `<tag>_actor` checkpoint format of RPO-LSTM/agent.py:136-147) and reproduce log-prob, entropy and LSTM state
    of a single step and of a 3-step sequence to 1e-6."""
    import os
    import torch
    from ouzelum_b200.rollout import RecurrentActor
    d = {}
    for f in ("rpo_lstm_actor.npz", "rpo_lstm_actor_sd_mlp.npz", "rpo_lstm_actor_sd_lstm.npz"):
        with np.load(os.path.join(os.path.dirname(__file__), "golden", f)) as z:
            d.update({k: z[k] for k in z.files})
    sd = {k[4:]: torch.from_numpy(d[k]) for k in d if k.startswith("sd__")}
    a = RecurrentActor()
    assert set(sd) == set(a.state_dict())                       # same parameter names and shapes as the reference module
    a.load_state_dict(sd, strict=True)
    t = lambda k: torch.from_numpy(d[k])
    B = d["h0"].shape[1]
    with torch.no_grad():
        for tag, obs, done in (("1", t("obs")[:B], t("done")[:B]), ("T", t("obs"), t("done"))):
            mean, std, (h, c) = a.distribution(obs, (t("h0"), t("c0")), done)
            logp, ent = a.log_prob_entropy(mean, std, t("a" + tag))          # the reference's sampled action under OUR distribution
            torch.testing.assert_close(logp, t("lp" + tag), rtol=1e-6, atol=2e-6)
            torch.testing.assert_close(ent, t("en" + tag), rtol=1e-6, atol=1e-6)
            torch.testing.assert_close(h, t("h" + tag), rtol=1e-6, atol=1e-6)
            torch.testing.assert_close(c, t("c" + tag), rtol=1e-6, atol=1e-6)
        # forward() has the reference's signature and return tuple: (action, log-prob, entropy, lstm_state)
        act, lp, en, st = a(t("obs")[:B], (t("h0"), t("c0")), t("done")[:B], action=t("a1"))
        assert act.shape == (B, 4) and lp.shape == (B,) and en.shape == (B,) and st[0].shape == (1, B, 128)
        torch.testing.assert_close(en, t("en1"), rtol=1e-6, atol=1e-6)


def test_c_abi_argument_errors_need_no_gpu(lib):
    """Argument validation happens before any CUDA call: non-zero return + a message in ozl_last_error()."""
    L = lib.lib
    msg = lambda: L.ozl_last_error().decode()
    assert L.ozl_step(None, None, None, None, None, None, None, None, None) != 0 and "env is NULL" in msg()
    assert L.ozl_step_host_sync(None, None, None) != 0 and "io is NULL" in msg()
    io = lib.OzlHostIo()
    assert L.ozl_step_host_sync(None, ctypes.byref(io), None) != 0 and "done_host is NULL" in msg()
    assert L.ozl_ekf_lee_landed_step(None, None, None, None, None, None, None, None, None, None) != 0 and "husky args are NULL" in msg()
    assert L.ozl_ekf_lee_step(None, None, None) != 0 and "NULL argument" in msg()
    assert L.ozl_rollout(None, 4, None, None, None, None, None) != 0 and "env is NULL" in msg()
    out = ctypes.c_uint64()
    assert L.ozl_get_step_count(None, ctypes.byref(out), None) != 0 and "env is NULL" in msg()
    assert L.ozl_cfg_default(None, 16) != 0 and "cfg is NULL" in msg()
    bad = lib.default_cfg(16)
    bad.abi_version = 999
    h = ctypes.c_void_p()
    assert L.ozl_create(ctypes.byref(bad), 0, ctypes.byref(h)) != 0 and "abi_version" in msg()
    # NVLink metrics exchange: rank / world validation and NULL handles
    x = ctypes.c_void_p()
    assert L.ozl_metrics_xchg_create(3, 2, 0, ctypes.byref(x)) != 0 and "rank 3 / world 2" in msg()
    assert L.ozl_metrics_xchg_create(0, 99, 0, ctypes.byref(x)) != 0 and "world 99" in msg()
    assert L.ozl_metrics_xchg_create(0, 1, 0, None) != 0 and "NULL argument" in msg()
    assert L.ozl_metrics_push(None, None, None, None, 0, None) != 0 and "NULL env" in msg()
    assert L.ozl_metrics_sum(None, None, None, None) != 0 and "NULL argument" in msg()
    assert L.ozl_metrics_xchg_ipc_handle(None, None) != 0 and "NULL argument" in msg()
    assert L.ozl_metrics_xchg_status(None, None, None, None, None) != 0 and "NULL exchange" in msg()


def test_compat_shims_resolve_the_reference_trainer_imports(lib, tmp_path):
    """ouzelum_b200.compat (SURVEY 8f rank 1): the module names a reference trainer imports resolve to this package's pieces;
    the gym stand-in has gym 0.24's Wrapper / ObservationWrapper semantics (what RPO-LSTM/utils.py:4-39 subclasses)."""
    import importlib
    import sys
    import ouzelum_b200
    from ouzelum_b200 import compat
    before = {k: sys.modules.get(k) for k in ("gym", "gym.spaces", "isaacgym", "isaacgymenvs", "isaacgymenvs.utils",
                                              "isaacgymenvs.utils.POMDP", "isaacgymenvs.tasks", "torch.utils.tensorboard")}
    try:
        installed = compat.install()
        assert {"isaacgym", "isaacgymenvs", "gym"} <= set(installed)             # none of them exists in this image (tensorboard does)
        import gym
        import isaacgym  # noqa: F401
        import isaacgymenvs
        from isaacgymenvs.utils.POMDP import POMDPWrapper
        from torch.utils.tensorboard import SummaryWriter
        assert isaacgymenvs.make is ouzelum_b200.make
        assert POMDPWrapper is importlib.import_module("ouzelum_b200.pomdp").POMDPWrapper
        SummaryWriter(str(tmp_path / "tb")).add_scalar("a", 1.0, 0)     # the real one if tensorboard is installed, else the no-op stand-in

        class Inner:
            num_envs, action_space = 3, gym.spaces.Box(-1.0, 1.0, (4,))

            def reset(self):
                return {"obs": "o0"}

            def step(self, a):
                return {"obs": a}, 1.0, False, {}

        class Extract(gym.ObservationWrapper):
            def observation(self, obs):
                return obs["obs"]

        class Count(gym.Wrapper):
            def __init__(self, env):
                super().__init__(env)
                self.n = 0

            def step(self, a):
                self.n += 1
                return self.env.step(a)
        e = Count(Extract(Inner()))
        assert e.reset() == "o0" and e.step("a1")[0] == "a1" and e.n == 1
        assert e.num_envs == 3 and isinstance(e.action_space, gym.spaces.Box) and e.action_space.shape == (4,)
        with pytest.raises(AttributeError):
            e.no_such_attribute
        assert compat.install() == []                                            # idempotent: nothing left to install
    finally:
        for k, v in before.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


_TRAINER_MAIN = '''
import argparse

import gym
import isaacgym  # noqa: F401
import isaacgymenvs
import torch
from isaacgymenvs.utils.POMDP import POMDPWrapper
from torch.utils.tensorboard import SummaryWriter

from agent import PPO

parser = argparse.ArgumentParser()
parser.add_argument("--env", default="Landing")
parser.add_argument("--num_envs", type=int, default=4096)
parser.add_argument("--POMDP", default="flicker")
parser.add_argument("--pomdp_prob", type=float, default=0.1)
parser.add_argument("--total_steps", type=int, default=30000000)
args = parser.parse_args()
assert (args.env, args.num_envs, args.POMDP, args.pomdp_prob) == ("Landing", 4096, "flicker", 0.1)
assert issubclass(PPO, gym.Wrapper) and SummaryWriter is not None
POMDP = POMDPWrapper(pomdp=args.POMDP, pomdp_prob=args.pomdp_prob)
# the call of RPO-LSTM/main.py:41 as SURVEY.md section 3.1 records it
envs = isaacgymenvs.make(seed=0, task="Landing", num_envs=4096, sim_device="cuda:0", rl_device="cuda:0", graphics_device_id=-1, headless=True, force_render=True)
'''

_TRAINER_AGENT = '''
import gym


class PPO(gym.Wrapper):
    pass
'''


def test_reference_trainer_reaches_make_through_the_compat_launcher(tmp_path):
    """A trainer laid out like the reference's RPO-LSTM/main.py (the same gym / isaacgym / isaacgymenvs / POMDP / tensorboard
    imports, `from agent import PPO` from a file beside it, the argparse flags and command line of SURVEY.md section 1, the
    make() call of section 3.1) through `python -m ouzelum_b200.compat`: every import resolves and the script gets as far as
    isaacgymenvs.make(), which refuses loudly because no CUDA device is visible to it (no CPU fallback)."""
    import subprocess
    import sys
    trainer = tmp_path / "trainer"
    trainer.mkdir()
    (trainer / "main.py").write_text(_TRAINER_MAIN)
    (trainer / "agent.py").write_text(_TRAINER_AGENT)
    r = subprocess.run([sys.executable, "-m", "ouzelum_b200.compat", str(trainer / "main.py"),
                        "--env", "Landing", "--num_envs", "4096", "--POMDP", "flicker", "--pomdp_prob", "0.1"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=300,
                       env={**os.environ, "PYTHONPATH": ROOT, "CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0
    assert "no CUDA device is visible and there is no CPU fallback" in r.stderr, r.stderr[-2000:]
    assert "isaacgymenvs.make" in r.stderr or "main.py" in r.stderr
