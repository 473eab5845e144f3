import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def built():
    """Build (or reuse) liboracle.so and libualm.so."""
    import pyoracle
    pyoracle.build()
    from uneven_planner_b200 import build as b
    b.build()
    return True


@pytest.fixture(scope="session")
def bumps_map(built):
    from uneven_planner_b200 import maps
    return maps.synthetic_terrain("bumps", seed=3)


# The reference's terrains are built from the reference project's point clouds, which are not part of this repository.  Where
# maps_built/<name>.umap cannot be had, a seeded synthetic terrain stands in for it (maps.terrain_or_standin), so every test that
# takes a terrain runs on a clean checkout.  On a stand-in those tests compare the CUDA path with the oracle, not anything with
# the reference's terrains.
@pytest.fixture(scope="session")
def hill_map(built):
    from uneven_planner_b200 import maps
    return maps.terrain_or_standin("hill")


@pytest.fixture(scope="session")
def terrain(built):
    """terrain(name) -> UnevenMapData of one of the reference's terrains, or its stand-in."""
    from uneven_planner_b200 import maps
    return maps.terrain_or_standin


@pytest.fixture(scope="session")
def golden():
    """golden(name, map) -> the frozen oracle outputs of tests/golden/ generated on exactly this map (make_golden.py).

    <name>_oracle_golden.npz were generated on the reference's terrains; <name>_standin_oracle_golden.npz on the stand-ins, by this
    repository's own oracle, so against those the oracle is only pinned to its earlier self (the CUDA path is still compared with
    it bit for bit).  A stand-in's hash rests on numpy's float64 exp / cos giving the same bits on every host before the cast to
    float32, the property bumps_map's fixed inputs already rely on; a host where they differ fails here, loudly, not silently."""
    import hashlib

    def get(name, m):
        sha = hashlib.sha256(m.cells.tobytes()).hexdigest()
        for fn in (f"{name}_oracle_golden.npz", f"{name}_standin_oracle_golden.npz"):
            gold = np.load(os.path.join(os.path.dirname(__file__), "golden", fn))
            if str(gold["map_sha256"]) == sha:
                return gold
        pytest.fail(f"no golden file of tests/golden/ was generated on this {name} map ({sha})")
    return get


@pytest.fixture(scope="session")
def oparams(built):
    import pyoracle as po
    from uneven_planner_b200 import _lib
    return po.params_from(_lib.default_params())
