#!/usr/bin/env python
"""Generates tests/golden/weighted_sampler.json and tests/golden/weighted_sampler_draws.npz from the
REFERENCE's own WeightedSampler (oracle/_ref/libvgref_sampler.so, compiled from the reference's
include/voxgraph/frontend/submap_collection/weighted_sampler{,_inl}.h by oracle/Makefile target
`ref`).  Needs the reference sources; the tests read only the stored fixtures."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as o  # noqa: E402

cases = []
rng = np.random.default_rng(7)
for name, w in (("uniform_1000", np.ones(1000, np.float32)),
                ("random_777", rng.uniform(0.01, 5.0, 777).astype(np.float32)),
                ("spiky_64", np.where(np.arange(64) % 7 == 0, 100.0, 0.001).astype(np.float32)),
                ("single", np.array([2.5], np.float32)),
                ("with_zeros_300", (rng.uniform(0, 1, 300) > 0.5).astype(np.float32) * 3.0 + np.float32(0))):
    if w.sum() == 0:
        continue
    s = o.RefWeightedSampler(w)
    first = s.draw(64)
    second = s.draw(64)     # the generator keeps advancing across calls (mutable member)
    cases.append({"name": name, "weights": [float(x) for x in w], "draw_0_64": first.tolist(),
                  "draw_64_128": second.tolist()})
out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "weighted_sampler.json")
json.dump({"source": "voxgraph::WeightedSampler<Item>::getRandomItem compiled from /root/reference "
                     "(libstdc++ std::mt19937 + uniform_real_distribution<double>)", "cases": cases},
          open(out, "w"))
print("wrote", out, len(cases), "cases")

# longer streams on larger inputs: 2000 draws from each of five weight vectors, a fifth of the items zero
rng = np.random.default_rng(11)
arrays = {}
sizes = (1, 2, 33, 1000, 20000)
for n in sizes:
    w = rng.uniform(0.0, 3.0, n).astype(np.float32)
    w[rng.integers(0, n, n // 5)] = 0.0
    if w.sum() == 0:
        w[0] = 1.0
    arrays["weights_%d" % n] = w
    arrays["draws_%d" % n] = o.RefWeightedSampler(w).draw(2000)
out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "weighted_sampler_draws.npz")
np.savez_compressed(out, sizes=np.array(sizes, np.int32), **arrays)
print("wrote", out, len(sizes), "weight vectors")
