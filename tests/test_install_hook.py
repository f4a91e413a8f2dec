"""happysim_b200.install(): the reference's own Simulation.run / ParallelRunner.run_replicas routed through the engine.

CPU part: the example's user-defined step profile (examples/queuing/m_m_1_queue.py:104-169) tabulates exactly
(replayed from its recorded answers, tests/golden/ref_example_step_profile.npz); with the reference importable
(REF_DIRS): models that do not lower fall through to the reference's Python loop unchanged; eligibility rules.
GPU part (tests/test_gpu_install.py): the stock-seeded README quick-start gives the reference's own numbers."""
import importlib.util
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIRS = [os.path.join(ROOT, "baseline", "_ref"), "/root/reference"]


def _reference():
    for d in REF_DIRS:
        if os.path.isdir(os.path.join(d, "happysimulator")):
            if d not in sys.path:
                sys.path.insert(0, d)
            import happysimulator
            return happysimulator
    pytest.skip("reference not importable (baseline/_ref not installed)")


def _example_module():
    path = "/root/reference/examples/queuing/m_m_1_queue.py"
    if not os.path.exists(path):
        pytest.skip("reference examples live in /root/reference only (build container)")
    spec = importlib.util.spec_from_file_location("ref_example_mm1_t", path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["ref_example_mm1_t"] = mod
    spec.loader.exec_module(mod)
    return mod


class _RecordedProfile:
    """The example's MetastableLoadProfile, answering from what the reference answered at the same times: runs of
    equal rate, first_s[i] <= t <= last_s[i] -> rate[i] (written by tests/golden/gen_example_profile_golden.py)."""

    def __init__(self):
        z = np.load(os.path.join(ROOT, "tests", "golden", "ref_example_step_profile.npz"))
        self.first, self.last, self.rate = z["first_s"], z["last_s"], z["rate"]

    def get_rate(self, time):
        t = time.to_seconds()
        i = int(np.searchsorted(self.first, t, side="right")) - 1
        assert i >= 0 and t <= self.last[i], f"the reference was not asked for the rate at t = {t!r}"
        return float(self.rate[i])


def test_example_step_profile_tabulates_exactly():
    import happysim_b200 as hs
    from happysim_b200 import Instant
    prof = _RecordedProfile()
    sp = hs.StepProfile.from_profile(prof, end_s=400.0)
    assert list(sp.breakpoints) == [25.0, 30.0, 35.0, 55.0, 60.0, 65.0, 76.0, 87.0, 98.0, 109.0]
    assert list(sp.rates) == [5.0, 15.0, 5.0, 9.0, 15.0, 9.0, 7.0, 6.0, 5.0, 4.0, 3.0]
    rng = np.random.default_rng(3)
    ts = np.concatenate([rng.uniform(0, 400, 20000), np.array(sp.breakpoints), np.nextafter(sp.breakpoints, 0), np.nextafter(sp.breakpoints, 1e9)])
    for t in ts:
        i = Instant.from_seconds(float(t))
        assert sp.get_rate(i) == prof.get_rate(i), t


def test_non_step_profile_is_rejected_not_approximated():
    import happysim_b200 as hs

    class Ramp:
        def get_rate(self, time):
            return 5.0 + time.to_seconds()
    with pytest.raises(hs.UnsupportedModelError):
        hs.StepProfile.from_profile(Ramp(), end_s=20.0)

    class TwoChangesInOneScanStep:
        def get_rate(self, time):
            t = time.to_seconds()
            return 9.0 if 1.0002 <= t < 1.0004 else 5.0
    with pytest.raises(hs.UnsupportedModelError):
        hs.lowering.step_table_from_profile(TwoChangesInOneScanStep(), scan_end_s=5.0, scan_step_s=1e-3)
    breaks, rates = hs.lowering.step_table_from_profile(TwoChangesInOneScanStep(), scan_end_s=5.0, scan_step_s=1e-4)
    assert breaks == [1.0002, 1.0004] and rates == [5.0, 9.0, 5.0]


def test_install_falls_through_for_models_that_do_not_lower():
    """The metastable example defines its own entity (MM1Server) and event provider: it cannot be lowered, so after
    install() it must run on the reference's own loop and give the reference's own (seeded) numbers."""
    _reference()
    import happysim_b200 as hs
    ex = _example_module()
    np.random.seed(7)            # the example seeds `random` only; its Poisson arrivals come from numpy's global stream
    want = ex.run_metastable_simulation(duration_s=12.0, drain_s=2.0, seed=7)
    hs.install()
    try:
        np.random.seed(7)
        got = ex.run_metastable_simulation(duration_s=12.0, drain_s=2.0, seed=7)
        st = hs.install_stats()
    finally:
        hs.uninstall()
    assert st["fallbacks"] >= 1 and "MM1Server" in st["last_fallback_reason"]
    assert got.summary.total_events_processed == want.summary.total_events_processed
    assert got.source_generated == want.source_generated and got.server.stats_processed == want.server.stats_processed


def test_eligibility_rules():
    hsim = _reference()
    from happysim_b200 import hook
    from happysimulator import Instant, Simulation, Sink, Source
    from happysimulator.components.server.server import Server
    from happysimulator.distributions.exponential import ExponentialLatency

    def build(**kw):
        sink = Sink()
        server = Server("Server", service_time=ExponentialLatency(0.1), downstream=sink)
        return Simulation(sources=[Source.poisson(rate=8, target=server)], entities=[server, sink], **kw)
    assert hook._eligible(build(end_time=Instant.from_seconds(5))) is None
    assert "auto-termination" in hook._eligible(build())
    assert "start_time" in hook._eligible(build(start_time=Instant.from_seconds(1), duration=5.0))
    sim = build(duration=5.0)
    _ = sim.control
    assert "control" in hook._eligible(sim)


def test_trace_fn_reproduces_the_global_generators():
    from happysim_b200 import hook
    import math
    random.seed(5); np.random.seed(5)
    fn = hook._trace_fn_from_states(np.random.get_state(), random.getstate())
    arr, svc = fn(6)
    assert [float(x) for x in arr[0]] == [-math.log(1.0 - np.random.random()) for _ in range(6)]
    assert [float(x) for x in svc[0]] == [-math.log(1.0 - random.random()) for _ in range(6)]
