import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import oracle
from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.solver import Summary
from helpers import load_oracle, load_engine, options_pair
sc = scenes.scene_test_ba(seed=0)
for lam0 in (1e-10,):
    kw = dict(max_num_iterations=25, threshold_cost_change=1e-9, threshold_step_size=1e-9, initial_lambda=lam0)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc); io, _ = o.solve(oo)
    of = load_oracle(sc); of.sizes()
    e = load_engine(sc, identical_internal=of.get_internal()); s = Summary(); e.solve(eo, s); ie = s.optimization_info_list
    for k,(a,b) in enumerate(zip(ie, io)):
        print(k, a.iteration_status, b.iteration_status, "%.3e" % (abs(a.cost-b.cost)/b.cost), "%.3e" % (abs(a.damping_term-b.damping_term)/b.damping_term))
    Te,Xe = e.get_internal(); To,Xo = o.get_internal()
    print("param diff", np.abs(Te-To).max(), np.abs(Xe-Xo).max())
