"""CPU-only check that the launch plans of kernels 1, 2, 5 and 6 (tile, threads, shared memory, splits, kernel choice,
workspace bytes, refusals and their messages, the effect of the kernel-selection and tiling overrides) are the ones
recorded in tests/golden/plan_info_all.json by tests/golden/make_golden_plans.py."""
import json
import os
import sys

import pytest

from golden_util import GOLDEN

sys.path.insert(0, GOLDEN)
import make_golden_plans      # noqa: E402


def _sm_count():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.get_device_properties(0).multi_processor_count
    except Exception:       # pragma: no cover
        pass
    return 148              # the planner's value when no device is visible


def test_launch_plans_match_the_recorded_ones():
    if _sm_count() != 148:
        pytest.skip('the recorded plans are for 148 SMs')
    want = json.load(open(os.path.join(GOLDEN, 'plan_info_all.json')))['plans']
    env0 = {var: os.environ.get(var) for var, _ in make_golden_plans.SWITCHES}
    got = make_golden_plans.record()
    assert {var: os.environ.get(var) for var in env0} == env0          # the overrides are restored
    assert sorted(got) == sorted(want)
    bad = [k for k in want if got[k] != want[k]]
    assert not bad, [(k, want[k], got[k]) for k in bad[:10]]
