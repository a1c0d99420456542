"""The critic kernel's results, bit for bit, against a recording of an earlier build (tests/golden/critic_schedule.py):
one critic step of every golden case through the Agent API, and LearnerEngine.step with in-kernel sampling and the
replay write folded into the critic step."""
import numpy as np
import pytest

from tests.golden.critic_schedule import ALL_CASES, ENGINE_CASES, NPZ, critic_step, engine_steps

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def recorded():
    with np.load(NPZ) as z:
        return {k: z[k] for k in z.files}


def _check(recorded, prefix, got):
    want = {k[len(prefix):]: v for k, v in recorded.items() if k.startswith(prefix)}
    assert sorted(got) == sorted(want)
    bad = [k for k in got if not np.array_equal(got[k], want[k])]
    assert not bad, f"{prefix}: differ from the recording: {bad}"


@pytest.mark.parametrize("name", list(ALL_CASES))
def test_critic_step_matches_recording(recorded, name):
    _check(recorded, f"critic/{name}/", critic_step(name))


@pytest.mark.parametrize("name", ENGINE_CASES)
def test_engine_step_matches_recording(recorded, name):
    _check(recorded, f"engine/{name}/", engine_steps(name))
