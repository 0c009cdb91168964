"""Host-side check of the traversal ALGORITHM the fast kernel runs (stackless bit-trail over the
heap-indexed tree, ray replacement, vote-postponed leaves): a lock-step 32-lane CPU model of
k_f_trace4 (tools/sim_warp.py) must finish every ray and agree with the oracle's exhaustive
Bvh.CheckHit on primitive ids -- for any refill / vote thresholds."""
import os
import sys

import numpy as np
import pytest

from tests.conftest import ROOT
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sim_warp  # noqa: E402
from mafrixraytracing_b200 import scenes  # noqa: E402
from oracle import oracle  # noqa: E402


@pytest.mark.parametrize("name,kw", [("c2_spot", dict(width=20, height=12)), ("cornell", dict(width=14, height=14)),
                                     ("c1_cube", dict(width=16, height=12))])
@pytest.mark.parametrize("refill_t,leaf_t", [(1, 1), (12, 16), (1, 32), (32, 4)])
def test_warp_model_finishes_and_matches_oracle(name, kw, refill_t, leaf_t):
    desc = scenes.WORKLOADS[name](**kw)
    sc = sim_warp.flatten(desc)
    uv = []
    rays = sim_warp.camera_rays(desc, seed=3, uv_out=uv)
    out, iters, stuck = sim_warp.run_warp(sc, rays, refill_t, leaf_t, max_iters=20000)
    assert stuck is None and len(out) == len(rays)
    prim, t = oracle.OracleScene(desc).trace_primary(np.array(uv))
    got = np.array([sc["ref"][sc["slots"][out[r][1]][-1]] if out[r][1] >= 0 else -1 for r in range(len(rays))])
    assert (got != prim).mean() <= 0.02        # f32 boxes/rays vs the f64 oracle: only edge-grazing rays may differ
    both = (got == prim) & (prim >= 0)
    tt = np.array([out[r][0] for r in range(len(rays))])
    assert np.allclose(tt[both], t[both], rtol=1e-4)


def test_warp_model_shadow_queries_terminate():
    desc = scenes.c2_spot(width=16, height=10)
    sc = sim_warp.flatten(desc)
    rays = [(o, d, 2.5) for (o, d, _) in sim_warp.camera_rays(desc)]
    out, iters, stuck = sim_warp.run_warp(sc, rays, 12, 16, ANY=True, max_iters=20000)
    assert stuck is None and len(out) == len(rays)
    o = oracle.OracleScene(desc)
    op, _, _ = o.hit([r[0] for r in rays], [r[1] for r in rays], 1e-6, 2.5)
    occl = np.array([out[r][1] >= 0 for r in range(len(rays))])
    assert (occl != (op >= 0)).mean() <= 0.02


def _own_tree_sim(workload, env=None, size=("96", "54")):
    import re
    import subprocess
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "tools", "own_tree_sim.py"), workload, *size],
                                  text=True, env=dict(os.environ, **(env or {})))
    occ = re.search(r"shadow rays, occluded: (\d+) rays; from the surface ([\d.]+) records ([\d.]+) tris \| from the light "
                    r"([\d.]+) records ([\d.]+) tris\s+\(answers that differ: (\d+)\)", out)
    tot = re.search(r"all: closest ([\d.]+) records \+ ([\d.]+) tris per ray.*?; shadow ([\d.]+) \+ ([\d.]+)", out)
    return [float(x) for x in occ.groups()], [float(x) for x in tot.groups()]


@pytest.mark.parametrize("workload", ["c2_spot", "cornell"])
def test_shadow_query_order_is_answer_invariant_and_cheaper_in_the_cpu_model(workload):
    """tools/own_tree_sim.cpp models the shipped own-tree traversal (it reproduces the GPU's record / triangle counters
    on C2).  A shadow query may visit its children in any order: the answers of the shipped farthest-first order, of
    the old nearest-first order and of the same rays traced from the light must be identical, and farthest-first must
    not fetch more records per shadow ray than nearest-first did."""
    occ_far, tot_far = _own_tree_sim(workload)
    occ_near, tot_near = _own_tree_sim(workload, {"SIM_ANY_NEAREST": "1"})
    assert occ_far[0] == occ_near[0] > 100              # the same rays are occluded whichever order finds the occluder
    assert occ_far[5] == 0 and occ_near[5] == 0         # ... and whichever end the ray is traced from
    assert tot_far[:2] == tot_near[:2]                  # closest-hit queries are untouched
    assert tot_far[2] <= tot_near[2] and tot_far[3] <= tot_near[3] * 1.02
    if workload == "c2_spot":
        assert 3.0 < tot_near[0] < 3.7 and 3.6 < tot_near[2] < 4.7     # the GPU measures 3.35 and 4.19 records per ray
        assert tot_far[2] < 0.9 * tot_near[2]
