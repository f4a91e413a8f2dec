"""Data / BucketedData mirrors against the reference's own answers (tests/golden/ref_instrumentation.npz, written by
tests/golden/gen_instrumentation_golden.py from the same seeded inputs) and against hand-checked values."""
import json
import os
import random

import numpy as np

import happysim_b200 as hs

REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_instrumentation.npz"))


def test_data_aggregations_hand_checked():
    d = hs.Data()
    d._samples = [(0.1, 1.0), (0.6, 3.0), (1.2, 2.0), (2.9, 10.0)]
    assert d.count() == 4 and d.sum() == 16.0 and d.mean() == 4.0 and d.min() == 1.0 and d.max() == 10.0
    assert d.percentile(0.0) == 1.0 and d.percentile(1.0) == 10.0 and d.percentile(0.5) == 2.5
    b = d.bucket(1.0)
    assert b.times() == [0.0, 1.0, 2.0] and b.counts() == [2, 1, 1] and b.sums() == [4.0, 2.0, 10.0]
    assert d.between(0.5, 2.0).raw_values() == [3.0, 2.0]
    assert d.rate(1.0).raw_values() == [2.0, 1.0, 1.0]
    assert hs.Data().mean() == 0.0 and hs.Data().percentile(0.9) == 0.0 and not hs.Data()


def test_data_matches_the_reference_class():
    rnd = random.Random(3)
    samples = sorted((rnd.random() * 30, rnd.expovariate(2.0)) for _ in range(2000))
    a = hs.Data()
    a._samples = list(samples)
    assert [getattr(a, f)() for f in ("mean", "min", "max", "count", "sum", "std")] == REF["data_aggregates"].tolist()
    assert [a.percentile(p) for p in (0.0, 0.5, 0.9, 0.99, 1.0)] == REF["data_percentiles"].tolist()
    assert json.loads(json.dumps(a.bucket(2.5).to_dict())) == json.loads(str(REF["data_bucket_json"]))
    assert json.loads(json.dumps(a.rate(5.0).values)) == json.loads(str(REF["data_rate_json"]))


def test_percentile_helper_equals_the_reference_helper_float_for_float():
    from happysim_b200.instrumentation import _percentile_sorted as mine
    rnd = random.Random(1)
    got = []
    for n in (0, 1, 2, 3, 7, 100, 1001):
        v = sorted(rnd.random() * 10 for _ in range(n))
        for p in (-1, 0, 1e-9, 0.25, 0.5, 0.99, 0.999, 1, 2, rnd.random(), rnd.random()):
            got.append(mine(v, p))
    want = REF["percentile_sorted"]
    assert np.array_equal(np.array(got, np.float64).view(np.int64), want.view(np.int64))
