"""The REFERENCE's own test files (unchanged, read from <ref_harness.REFERENCE_ROOT>/tests) run against this repo's host-side
drop-in classes, served under the reference's module names by tests/ref_alias/ref_alias_plugin.py. These are the reference tests
that need no device: reward machine (4 files), spec io / completion / rewards / summary, encoders, agent plumbing, event contexts."""
import os
import subprocess
import sys

import pytest
from ref_harness import REFERENCE_MISSING, REFERENCE_ROOT

REF_TESTS = os.path.join(REFERENCE_ROOT, "tests")
FILES = ["test_reward_machine.py", "test_reward_machine_api.py", "test_reward_machine_extras.py", "test_reward_machine_shaping.py",
         "test_rmspec_io.py", "test_rmgen_completion.py", "test_rmgen_rewards.py", "test_rmspec_summary.py",
         "test_state_encoder_frozen_lake.py", "test_utils_encoding.py", "test_agent_rl.py", "test_agent_rl_actions.py",
         "test_officeworld_event_context.py", "test_frozenlake_event_context.py"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = [pytest.mark.reference, pytest.mark.skipif(not os.path.isdir(REF_TESTS), reason=REFERENCE_MISSING)]


def test_reference_host_side_tests_pass_on_the_dropin_classes():
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests", "ref_alias")]))
    cmd = [sys.executable, "-m", "pytest", "-p", "ref_alias_plugin", "-q", "-p", "no:cacheprovider", "--rootdir", REF_TESTS,
           "-c", os.devnull] + [os.path.join(REF_TESTS, f) for f in FILES]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd="/tmp", timeout=600)
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0, tail
    assert "29 passed" in res.stdout and "failed" not in res.stdout and "error" not in res.stdout.lower(), tail
