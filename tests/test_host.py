"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, the host
mirror keeps the reference's names / argument meaning / error behaviour, and the product fails loudly
without a CUDA device.  No compute calls are made here."""
import ctypes as C
import re
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    from twisterl_b200 import _lib
    L = _lib.load()
    header = (ROOT / "include" / "twisterl_b200.h").read_text()
    declared = set(re.findall(r"\b(twr_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/twisterl_b200.h but not exported"
    assert declared == set(_lib.SYMBOLS)
    assert L.twr_abi_version() == _lib.ABI_VERSION == 3


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import twisterl_b200 as tw
    assert tw._lib.load().twr_device_count() == 0
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tw.Engine()
    p = tw.env.Puzzle(3, 3, 2, 2, 256)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        p.reset()


def test_product_never_imports_the_oracle():
    for f in list((ROOT / "twisterl_b200").rglob("*.py")) + list((ROOT / "twisterl_b200" / "csrc").glob("*")):
        txt = f.read_text()
        assert "oracle" not in txt.replace("oracle/twr_oracle.h", "").replace("the oracle's libm", ""), f


def test_env_description_without_device():
    import twisterl_b200 as tw
    p = tw.env.Puzzle(4, 4, 1, 2, 256)
    assert p.obs_shape() == [16, 16] and p.num_actions() == 4 and p.twists() == ([], [])
    p.difficulty = 7
    assert p.difficulty == 7
    g = tw.env.GridWorld(5, 5, 64, 99)
    assert g.difficulty == 10 and g.obs_shape() == [25, 25]          # clamp to W+H (lib.rs:36)
    g.difficulty = 3
    assert g.difficulty == 3
    with pytest.raises(OverflowError):
        tw.env.Puzzle(-1, 3, 1, 1, 1)
    s = tw.env.spec_from_env(p)
    assert (s.kind, s.width, s.height, s.difficulty, s.depth_slope, s.max_depth) == (0, 4, 4, 7, 2, 256)
    with pytest.raises(TypeError, match="__extract_env__"):
        tw.env.spec_from_env(object())

    class Fake:
        def __extract_env__(self):
            return 12345
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tw.env.spec_from_env(Fake())


def test_pyenv_wrapper_is_rejected_by_collectors():
    import twisterl_b200 as tw

    class Dummy:                      # the reference's pure-Python DummyEnv (tests/test_all.py:14-29)
        def num_actions(self): return 2
        def obs_shape(self): return [2]
        def reset(self, d): self.d = d
        def observe(self): return [0]
        def masks(self): return [True, True]
        def is_final(self): return True
        def value(self): return 1.0
        def next(self, a): pass
        def set_state(self, s): pass
    e = tw.env.PyEnv(Dummy())
    assert e.num_actions() == 2 and e.obs_shape() == [2] and e.twists() == ([], [])
    e.reset()
    assert e.observe() == [0] and e.is_final() and e.reward() == 1.0
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tw.env.spec_from_env(e)


def test_ppo_collector_constructor_keywords():
    import twisterl_b200 as tw
    cfg = {"num_cores": 32, "num_episodes": 1024, "lambda": 0.995, "gamma": 0.99}   # examples/*.json "collecting"
    c = tw.collector.PPOCollector(**cfg)
    assert (c.num_episodes, c.gamma, c.lambda_, c.num_cores) == (1024, 0.99, 0.995, 32)
    c2 = tw.collector.PPOCollector(8, 0.9, 0.95, 1)
    assert (c2.num_episodes, c2.gamma, c2.lambda_, c2.num_cores) == (8, 0.9, 0.95, 1)
    with pytest.raises(TypeError):
        tw.collector.PPOCollector(8, 0.9, 0.95, 1, seed=3)
    with pytest.raises(TypeError):
        tw.collector.PPOCollector(8, 0.9)
    az = tw.collector.AZCollector(num_episodes=4, num_mcts_searches=8, C=1.4, max_expand_depth=2, num_cores=1)
    assert (az.num_episodes, az.num_mcts_searches, az.C, az.max_expand_depth, az.num_cores) == (4, 8, 1.4, 2, 1)
    with pytest.raises(TypeError):                      # AZ_CONFIG's stray "seed" key is rejected like in the reference
        tw.collector.AZCollector(num_episodes=4, num_mcts_searches=8, C=1.4, max_expand_depth=2, num_cores=1, seed=123)
    with pytest.raises(TypeError):
        az.collect(None, None)


def test_collected_data_mirror():                     # python_interface/collector.rs:24-137
    import twisterl_b200 as tw
    CD = tw.collector.CollectedData
    d1 = CD([[0]], [[0.1]], [0.2], [0.3], [1], [0])
    d2 = CD([[1]], [[0.4]], [0.5], [0.6], [0])
    assert d2.perms == [-1]
    d1.set_additional_data_item("rets", [1.0]); d2.set_additional_data_item("rets", [2.0])
    d2.merge(d1)                                       # collector.rs:101-126: d2 first, then d1
    assert d2.actions == [0, 1] and d2.obs == [[1], [0]] and d2.perms == [-1, 0]
    assert d2.additional_data == {"rets": [2.0, 1.0]} and d2.get_additional_data_item("nope") is None
    d2.perms = [None, 3]
    assert d2.perms == [-1, 3]
    d2.values = [9.0, 8.0]
    assert d2.values == [9.0, 8.0]
    a = CD(np.zeros((2, 3), np.uint16), np.zeros((2, 4), np.float32), np.zeros(2, np.float32), np.zeros(2, np.float32),
           np.zeros(2, np.uint8), np.full(2, -1, np.int8))
    assert a.obs == [[0, 0, 0], [0, 0, 0]] and a.perms == [-1, -1] and isinstance(a.obs, list)


def test_nn_mirror_layouts():                         # python_interface/layers.rs, nn/utils.py:17-59
    import twisterl_b200 as tw
    l = tw.nn.Linear([1, 2, 3, 4, 5, 6], [0, 0], True)
    assert (l.in_, l.out, l.apply_relu) == (3, 2, True)
    with pytest.raises(ValueError):
        tw.nn.Linear([1, 2, 3], [0, 0], False)
    e = tw.nn.EmbeddingBag([[1, 2], [3, 4], [5, 6]], [0, 0], True, [3], 0)
    p = tw.nn.Policy(e, tw.nn.Sequential([tw.nn.Linear([1] * 8, [0] * 4, True)]),
                     tw.nn.Sequential([tw.nn.Linear([1] * 16, [0] * 4, False)]),
                     tw.nn.Sequential([tw.nn.Linear([1] * 4, [0], False)]), [], [])
    d = p.desc()
    assert (d.obs_size, d.emb_size, d.n_common, d.n_action, d.n_value, d.n_perms) == (3, 2, 1, 1, 1, 0)
    assert d.common[0].in_ == 2 and d.common[0].out == 4 and d.action_net[0].out == 4
    with pytest.raises(TypeError):
        tw.nn.Sequential([1])


def test_install_as_twisterl_registers_reference_names():
    import twisterl_b200 as tw
    mod = tw.install_as_twisterl()
    import importlib
    assert importlib.import_module("twisterl.twisterl") is mod
    for sub, names in {"env": ["Puzzle", "PyBaseEnv", "PyEnv"], "nn": ["Linear", "EmbeddingBag", "Sequential", "Policy"],
                       "collector": ["PPOCollector", "AZCollector", "CollectedData", "solve", "evaluate"]}.items():
        for n in names:
            assert hasattr(getattr(mod, sub), n), (sub, n)
    assert importlib.import_module("grid_world").GridWorld is tw.env.GridWorld


def test_max_records_and_spec_validation():
    import ctypes as C
    from twisterl_b200 import _lib
    L = _lib.load()
    s = _lib.EnvSpec(0, 4, 4, 128, 2, 256)
    assert L.twr_max_records(C.byref(s), 65536) == 65536 * 257
    g = _lib.EnvSpec(1, 5, 5, 10, 0, 64)
    assert L.twr_max_records(C.byref(g), 10) == 650
    big = _lib.EnvSpec(0, 5, 5, 1, 1, 1)
    assert L.twr_max_records(C.byref(big), 1) == -1
    assert b"16 cells" in L.twr_last_error()


def test_reference_python_half_builds_on_this_module():
    """Drop-in check that needs a checkout of the reference, AI4quantum/twisteRL (helpers.reference_checkout; skipped
    without one): with twisterl_b200 installed as `twisterl.twisterl`, the reference's own unmodified Python half
    (twisterl.utils.load_config / prepare_algorithm, BasicPolicy.to_rust) builds PPO and AlphaZero from its own
    JSON configs and hands our nn.Policy / collectors the layouts they expect.  No device is touched."""
    import subprocess
    import sys
    from helpers import reference_checkout
    ref = reference_checkout()
    if ref is None:
        pytest.skip("no checkout of the reference (set TWISTERL_REFERENCE or stage one under oracle/_ref/reference)")
    code = r'''
import sys, json
sys.path.insert(0, %r)
import twisterl_b200
twisterl_b200.install_as_twisterl()
sys.path.insert(0, %r)
from twisterl.utils import load_config, prepare_algorithm
out = {}
for name in ("ppo_puzzle8_v1", "ppo_puzzle15_v1"):
    algo = prepare_algorithm(load_config(%r %% name))
    pol = algo.policy.to_rust()
    out[name] = [type(algo).__name__, type(algo.env).__module__, type(algo.collector).__module__, type(pol).__module__,
                 int(pol.embeddings.vectors.shape[0]), int(pol.embeddings.bias.size), int(pol.num_actions),
                 algo.env.obs_shape(), algo.env.num_actions()]
# the reference trainer's own data_to_torch / train_step (rl/ppo.py:25-106) on a CollectedData of this module
import numpy as np
from twisterl_b200.collector import CollectedData
R = 6
rng = np.random.default_rng(0)
obs = np.arange(16)[None, :] * 16 + rng.integers(0, 16, size=(R, 16))
d = CollectedData(obs.astype(np.uint16), rng.standard_normal((R, 4)).astype(np.float32), np.zeros(R, np.float32),
                  np.zeros(R, np.float32), rng.integers(0, 4, R).astype(np.uint8), np.full(R, -1, np.int8))
d.set_additional_data_item("advs", rng.standard_normal(R).astype(np.float32))
d.set_additional_data_item("rets", rng.standard_normal(R).astype(np.float32))
td = algo.data_to_torch(d)
td = td[0] if isinstance(td[0], tuple) else td
out["torch_shapes"] = [list(t.shape) for t in td]
algo.train_step(td)
print(json.dumps(out))
''' % (str(ROOT), str(ref / "src"), str(ref / "examples" / "%s.json"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["ppo_puzzle8_v1"] == ["PPO", "twisterl_b200.env", "twisterl_b200.collector", "twisterl_b200.nn", 81, 512, 4, [9, 9], 4]
    assert out["ppo_puzzle15_v1"] == ["PPO", "twisterl_b200.env", "twisterl_b200.collector", "twisterl_b200.nn", 256, 512, 4, [16, 16], 4]
    assert out["torch_shapes"] == [[6, 256], [6], [6], [6], [6], [6]]


def test_balanced_schedule_host_model():
    """scripts/sim_balance.py restates `struct Sched` of twr_forward_tc2.cu on the host: every (group, step) item is
    issued exactly once, a pair never issues the same group twice within two items, hand-offs cannot deadlock, and the
    benchmark shape (256 groups, 74 pairs, 32 steps) costs 111 item slots instead of 128."""
    import importlib.util
    import random
    spec = importlib.util.spec_from_file_location("sim_balance", ROOT / "scripts" / "sim_balance.py")
    sb = importlib.util.module_from_spec(spec)
    argv = sys.argv
    sys.argv = ["sim_balance.py"]
    try:
        spec.loader.exec_module(sb)
    finally:
        sys.argv = argv
    assert sb.check(256, 74, 32, 2) == (111.0, 111)
    assert sb.check(256, 74, 32, 0) == (128.0, 128)
    assert sb.check(256, 74, 128, 2)[1] == 3 * 128 + 59          # the adaptive 128-step launches: ceil(34 * 128 / 74) extra slots
    rng = random.Random(3)
    for _ in range(300):
        sb.check(rng.randint(1, 700), rng.choice([2, 7, 66, 74]), rng.randint(1, 40), 2)


def test_header_is_plain_c_and_links(tmp_path):
    """include/twisterl_b200.h must be usable from C (the drop-in boundary is a C ABI): compile a C99 translation unit
    against it with -pedantic, link the shared library and call an entry point that needs no device."""
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("gcc not available")
    src = tmp_path / "abi.c"
    src.write_text('#include "twisterl_b200.h"\n#include <stdio.h>\n'
                   'int main(void) { twr_env_spec s = {0, 4, 4, 1, 2, 256}; printf("%d %lld\\n", twr_abi_version(), '
                   '(long long)twr_max_records(&s, 10)); return twr_abi_version() == TWR_ABI_VERSION ? 0 : 1; }\n')
    libdir = ROOT / "twisterl_b200" / "lib"
    exe = tmp_path / "abi"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", f"-I{ROOT / 'include'}", str(src),
                        f"-L{libdir}", "-ltwisterl_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.split() == ["3", "30"], (r.stdout, r.stderr)   # 10 episodes x (2*1 + 1) records


def test_safetensors_reader_rejects_corrupt_headers(tmp_path):
    """The native checkpoint reader treats the header as untrusted file content: negative / overflowing dimensions,
    offsets outside the file and shape/offset mismatches come back as TWR_ERR_INVALID (never an exception or a wild
    allocation across the C boundary).  Parsing happens before the engine is touched, so a placeholder handle is enough."""
    import json
    import struct
    from twisterl_b200 import _lib
    L = _lib.load()
    fake_engine = C.create_string_buffer(64)

    def write(name, header, payload=b"\0" * 64):
        js = json.dumps(header).encode()
        p = tmp_path / name
        p.write_bytes(struct.pack("<Q", len(js)) + js + payload)
        return str(p).encode()

    cases = {
        "neg.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [-4, -4], "data_offsets": [0, 64]}},
        "huge.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [2 ** 31, 2 ** 31], "data_offsets": [0, 64]}},
        "overflow.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [2 ** 30, 2 ** 30, 2 ** 30], "data_offsets": [0, 64]}},
        "past_end.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [4, 4], "data_offsets": [1 << 40, (1 << 40) + 64]}},
        "reversed.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [4, 4], "data_offsets": [64, 0]}},
        "mismatch.safetensors": {"embeddings.weight": {"dtype": "F32", "shape": [4, 5], "data_offsets": [0, 64]}},
        "f16.safetensors": {"embeddings.weight": {"dtype": "F16", "shape": [4, 8], "data_offsets": [0, 64]}},
    }
    for name, hdr in cases.items():
        h = C.c_void_p()
        rc = L.twr_policy_create_from_safetensors(fake_engine, write(name, hdr), None, 0, 0, None, None, 0, C.byref(h))
        assert rc in (-1, -2) and not h.value, (name, rc)
        assert L.twr_last_error(), name
    (tmp_path / "short.safetensors").write_bytes(b"\x10\0\0\0\0\0\0\0{")
    h = C.c_void_p()
    assert L.twr_policy_create_from_safetensors(fake_engine, str(tmp_path / "short.safetensors").encode(), None, 0, 0, None, None, 0, C.byref(h)) == -1


def test_puzzle_opt_in_twists_are_a_symmetry():
    """`Puzzle(..., add_perms=True)` hands the policy the {identity, transpose} twist set (SURVEY.md 8a row T): a pair of
    permutations for which twist(step(s, a)) == step(twist(s), A(a)) on the oracle env, with the solved board fixed."""
    import twisterl_b200 as tw
    from helpers import transpose_twists
    from oracle import orc
    assert tw.env.Puzzle(4, 4, 1, 2, 256).twists() == ([], [])
    assert tw.env.Puzzle(4, 3, 1, 2, 256, add_perms=True).twists() == ([], [])           # square boards only
    obs_perms, act_perms = tw.env.Puzzle(4, 4, 1, 2, 256, add_perms=True).twists()
    assert (obs_perms, act_perms) == tuple(transpose_twists(4))
    assert sorted(obs_perms[1]) == list(range(256)) and obs_perms[0] == list(range(256))
    rng = np.random.default_rng(0)
    env, tenv = orc.Env(orc.puzzle_spec(4, 4, 1, 2, 256)), orc.Env(orc.puzzle_spec(4, 4, 1, 2, 256))
    twist_state = lambda obs: [v % 16 for v in sorted(obs_perms[1][o] for o in obs)]      # obs index -> (cell, tile) under the twist
    assert twist_state(env.observe()) == env.get_state()                                   # solved board is a fixed point
    for _ in range(300):
        a = int(rng.integers(0, 4))
        tenv.set_state(twist_state(env.observe()))
        env.step(a); tenv.step(act_perms[1][a])
        assert twist_state(env.observe()) == tenv.get_state()
