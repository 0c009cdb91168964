"""The batch z-test of tests/test_gpu_path_parity.py (the fast path's default sampler against the f64 renderer) run on
the CPU oracle alone, at fewer paths: two seeds of the same renderer must pass it, and the same renderer with the
scene's albedo 1 % higher must fail it.  So the test is neither vacuous nor flaky, and this needs no GPU."""
import numpy as np

from oracle import oracle
from .test_gpu_path_parity import SKY_MATERIALS, Z_FRAME, Z_TILE, batch_means, sky_material_scene, z_scores

W, H, BATCHES, SPP = 80, 50, 32, 4


def _batches(desc, seed):
    o = oracle.OracleSkyScene(desc)
    return batch_means(lambda n, k: o.sample(n, seed=seed, first_sample=k), BATCHES, SPP, W, H)


def test_batch_z_test_passes_two_seeds_and_fails_a_one_percent_albedo_change():
    desc = sky_material_scene(SKY_MATERIALS["constant"], width=W, height=H)
    ref = _batches(desc, seed=1)
    z, zt, se = z_scores(_batches(desc, seed=2), ref)
    assert abs(z) <= Z_FRAME and zt <= Z_TILE, (z, zt)
    brighter = sky_material_scene(("lambert", tuple(1.01 * np.array(SKY_MATERIALS["constant"][1]))), width=W, height=H)
    z1, zt1, _ = z_scores(_batches(brighter, seed=2), ref)
    assert abs(z1) > Z_FRAME, (z1, se)
    print(f"two seeds: z {z:+.2f}, worst tile {zt:.2f}; albedo x1.01: z {z1:+.2f}, worst tile {zt1:.2f}; relative SE {se:.1e}")
