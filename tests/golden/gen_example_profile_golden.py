"""Answers of the reference example's own step profile (examples/queuing/m_m_1_queue.py, MetastableLoadProfile):

    HS_REFERENCE_ROOT=<checkout of happy-simulator> python tests/golden/gen_example_profile_golden.py

-> tests/golden/ref_example_step_profile.npz.  The profile is asked at every time StepProfile.from_profile(...,
end_s=400) scans and at every time tests/test_install_hook.py checks; its answers, sorted by time, are stored as runs
of equal rate (first_s[i] <= t <= last_s[i] -> rate[i]), which keeps every answer and nothing else."""
import importlib.util
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ["HS_REFERENCE_ROOT"]
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), REF]

import happysim_b200 as hs  # noqa: E402
from happysimulator import Instant  # noqa: E402

spec = importlib.util.spec_from_file_location("ref_example_mm1", os.path.join(REF, "examples", "queuing", "m_m_1_queue.py"))
ex = importlib.util.module_from_spec(spec)
sys.modules["ref_example_mm1"] = ex
spec.loader.exec_module(ex)
prof = ex.MetastableLoadProfile()
seen = {}


class Recorder:
    def get_rate(self, time):
        t = time.to_seconds()
        seen[t] = float(prof.get_rate(Instant.from_seconds(t)))
        return seen[t]


sp = hs.StepProfile.from_profile(Recorder(), end_s=400.0)
rng = np.random.default_rng(3)        # the check times of test_example_step_profile_tabulates_exactly
ts = np.concatenate([rng.uniform(0, 400, 20000), np.array(sp.breakpoints), np.nextafter(sp.breakpoints, 0),
                     np.nextafter(sp.breakpoints, 1e9)])
for t in ts:
    seen[Instant.from_seconds(float(t)).to_seconds()] = float(prof.get_rate(Instant.from_seconds(float(t))))

first, last, rate = [], [], []
for t in sorted(seen):
    if rate and seen[t] == rate[-1]:
        last[-1] = t
    else:
        first.append(t); last.append(t); rate.append(seen[t])
np.savez_compressed(os.path.join(HERE, "ref_example_step_profile.npz"), first_s=np.array(first), last_s=np.array(last),
                    rate=np.array(rate))
print(len(seen), "answers in", len(rate), "runs")
