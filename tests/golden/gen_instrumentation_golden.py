"""Known answers of the reference's instrumentation/data.py on fixed seeded inputs:

    HS_REFERENCE_ROOT=<checkout of happy-simulator> python tests/golden/gen_instrumentation_golden.py

-> tests/golden/ref_instrumentation.npz: what the UNMODIFIED reference's Data (aggregations, percentiles,
bucket(), rate()) and _percentile_sorted answer for the inputs tests/test_instrumentation.py draws from the same
seeds.  The test compares the host mirrors (happy-simulator_b200/instrumentation.py) with them, floats bitwise."""
import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.environ["HS_REFERENCE_ROOT"])

from happysimulator.instrumentation.data import Data, _percentile_sorted  # noqa: E402

out = {}

# test_data_matches_the_reference_class
rnd = random.Random(3)
samples = sorted((rnd.random() * 30, rnd.expovariate(2.0)) for _ in range(2000))
d = Data()
d._samples = list(samples)
out["data_aggregates"] = np.array([getattr(d, f)() for f in ("mean", "min", "max", "count", "sum", "std")], np.float64)
out["data_percentiles"] = np.array([d.percentile(p) for p in (0.0, 0.5, 0.9, 0.99, 1.0)], np.float64)
out["data_bucket_json"] = np.array(json.dumps(d.bucket(2.5).to_dict()))
out["data_rate_json"] = np.array(json.dumps(d.rate(5.0).values))

# test_percentile_helper_equals_the_reference_helper_float_for_float
rnd = random.Random(1)
answers = []
for n in (0, 1, 2, 3, 7, 100, 1001):
    v = sorted(rnd.random() * 10 for _ in range(n))
    for p in (-1, 0, 1e-9, 0.25, 0.5, 0.99, 0.999, 1, 2, rnd.random(), rnd.random()):
        answers.append(_percentile_sorted(v, p))
out["percentile_sorted"] = np.array(answers, np.float64)

np.savez_compressed(os.path.join(HERE, "ref_instrumentation.npz"), **out)
print({k: v.shape for k, v in out.items()})
