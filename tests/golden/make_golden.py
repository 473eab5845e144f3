"""Generates tests/golden/<terrain>_oracle_golden.npz: frozen outputs of the CPU oracle for seeded problems on the
reference's terrains with the parameter sets of BASELINE.json's configs (uneven_planner_b200/configs.py).  Those need
maps_built/*.umap, built from the reference's .pcd clouds by __graft_entry__.build().  Where a terrain is absent it writes
<terrain>_standin_oracle_golden.npz instead, on the seeded synthetic terrain the tests use in its place
(maps.terrain_or_standin); those pin the oracle to itself, not to the reference.  The same numbers are what the CUDA path must
reproduce bit for bit."""
import hashlib, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyoracle as po
from uneven_planner_b200 import configs, maps, problems

B, SEED = 12, 0
for name in (sys.argv[1:] or ["hill", "desert", "volcano", "forest"]):
    m = maps.terrain_or_standin(name)
    kind = "" if maps.get_terrain(name, build_if_missing=False) is not None else "_standin"
    pb = problems.generate(m, B, seed=SEED, **configs.gen_kwargs(name))
    prm = po.params_from(configs.params_for(name))
    out = po.solve_batch(prm, po.OracleMap(m), pb, threads=4)
    np.savez_compressed(os.path.join(HERE, f"{name}{kind}_oracle_golden.npz"),
                        B=B, seed=SEED, map_sha256=hashlib.sha256(m.cells.tobytes()).hexdigest(),
                        N=pb.N, M=pb.M, ret_code=np.array([r[0].ret_code for r in out]), n_evals=np.array([r[0].n_evals for r in out]),
                        outer_iters=np.array([r[0].outer_iters for r in out]), inner_cost=np.array([r[0].inner_cost for r in out]),
                        c_xy=np.concatenate([r[1] for r in out]), c_yaw=np.concatenate([r[2] for r in out]))
    print("wrote golden for", B, "problems on", name, m.name)
