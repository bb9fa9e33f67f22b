"""Acceptance on the reference's own code (needs a checkout of AI4quantum/twisteRL and a GPU; skipped otherwise).

With `twisterl_b200.install_as_twisterl()` standing in for the Rust extension, (1) the reference's own pytest files
tests/test_all.py, tests/test_utils.py and tests/test_custom_env_integration.py pass, and (2) the reference's UNMODIFIED
trainer -- `twisterl.utils.prepare_algorithm(load_config("examples/ppo_puzzle8_v1.json")).learn(n)`, i.e. what
`python -m twisterl.train` runs (src/twisterl/train.py:21-41) -- trains on this engine far enough for its curriculum to
raise the difficulty, as does the same object after `twisterl_b200.accelerate()` (device hand-off + device weight sync).

The checkout is $TWISTERL_REFERENCE, else a copy staged under the git-ignored oracle/_ref/reference (helpers.reference_checkout).
Nothing here is read by the product or by the other tests."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

from helpers import reference_checkout

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu


def _reference():
    ref = reference_checkout()
    if ref is None:
        pytest.skip("no checkout of the reference (set TWISTERL_REFERENCE or stage one under oracle/_ref/reference)")
    return ref


PRELUDE = """
import sys
sys.path.insert(0, {root!r})
import twisterl_b200
twisterl_b200.configure(device=0, precision={precision!r}, seed=7)
twisterl_b200.install_as_twisterl()
sys.path.insert(0, {src!r})
"""


def _python(code, ref, precision="f16x2w16", timeout=900):
    full = PRELUDE.format(root=str(ROOT), precision=precision, src=str(ref / "src")) + code
    return subprocess.run([sys.executable, "-c", full], capture_output=True, text=True, timeout=timeout, cwd="/tmp")


def test_reference_own_test_files_pass_on_this_engine():
    ref = _reference()
    files = [str(ref / "tests" / f) for f in ("test_all.py", "test_utils.py", "test_custom_env_integration.py")]
    # test_pull_new_hub_model needs the pytest-mock plugin (not in this image) and the network
    code = f"import pytest\nsys.exit(pytest.main({files!r} + ['-q', '-p', 'no:cacheprovider', '--rootdir', '/tmp', '-k', 'not test_pull_new_hub_model']))\n"
    r = _python(code, ref)
    tail = (r.stdout[-3000:] + r.stderr[-2000:])
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout.splitlines()[-1], tail


TRAIN = """
import json, time, torch
from twisterl.utils import load_config, prepare_algorithm
config = load_config({cfg!r})
config["algorithm"]["device"] = "cuda"
config["algorithm"]["logging"] = {{"log_freq": 0, "checkpoint_freq": 0}}
torch.manual_seed(0)
algo = prepare_algorithm(config)
assert type(algo.collector).__module__ == "twisterl_b200.collector" and type(algo.env).__module__ == "twisterl_b200.env"
{accelerate}
t0 = time.time()
algo.learn({steps})
(times, bench, train), _ = algo.learn_step()
print(json.dumps({{"difficulty": int(algo.env.difficulty), "seconds": time.time() - t0, "success": bench["success"],
                  "times": {{k: float(v) for k, v in times.items()}}}}))
"""


@pytest.mark.parametrize("accelerated", [False, True])
def test_reference_trainer_learns_on_this_engine(accelerated):
    ref = _reference()
    code = TRAIN.format(cfg=str(ref / "examples" / "ppo_puzzle8_v1.json"), steps=40,
                        accelerate="twisterl_b200.accelerate(algo)" if accelerated else "")
    r = _python(code, ref)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    print(("accelerated " if accelerated else "unmodified ") + json.dumps(out))
    assert out["difficulty"] >= 3, out             # the curriculum advanced: evaluate / collect / train all did their part
    if accelerated:                                # no host round trip left in these two
        assert out["times"]["to_rust"] < 0.005 and out["times"]["data_to_torch"] < 0.005, out
