#!/usr/bin/env python
"""Round-2 fixtures, generated from the REFERENCE ITSELF (needs OFB_REFERENCE_DIR naming a checkout of the original
project; the tests only read the committed file): tests/golden/velocity_golden_r2.npz.

* module_*   : the inline least-squares system of optical_flow_experiments/of_module.py:136-146. The statements
  (A = ..., B = ..., the `for` loop, `np.linalg.lstsq(A, B)`) are AST-extracted from the script's `while` body and exec'd
  unmodified on seeded inputs; the per-point distances come from the 4-argument of.r_tilde of
  sensor_precision_experiments/pixhawk_pure_IMU/of_library.py:365-384 (AST-extracted as well), as at of_module.py:125.
* te_*       : the time-evolution sweep, simulation.py:472-501. The block is commented out in the reference (a module
  level string); its text is parsed and its statements are exec'd unmodified with the reference's own
  generate_test_data / of_simulation. The block prints `data` after every step, so a print hook records the trajectory.
* live_*     : the only LIVE section of simulation.py, lines 753-774 (moving points + parallel plane), exec'd
  statement by statement after the module's own globals (122, 154-178) with np.random seeded; two seeds, so the tests
  can scale their tolerance with the reference's own sampling noise.
"""
import ast
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
REF = ref_loader.REF


def module_statements():
    """[A = ..., B = ..., for ...: ..., v_obs,R,rank,s = np.linalg.lstsq(A,B)] of of_module.py:136-146"""
    src = open(os.path.join(REF, "optical_flow_experiments", "of_module.py")).read()
    tree = ast.parse(src)
    loop = next(n for n in ast.walk(tree) if isinstance(n, ast.While))
    keep = []
    for st in loop.body:
        seg = ast.get_source_segment(src, st)
        if isinstance(st, ast.Assign) and seg.startswith(("A = np.empty", "B = np.empty", "v_obs,R,rank,s")):
            keep.append(st)
        elif isinstance(st, ast.For) and "feasible_new" in seg and "ai" in seg:
            keep.append(st)
    assert len(keep) == 4, [ast.get_source_segment(src, k)[:40] for k in keep]
    return compile(ast.Module(body=keep, type_ignores=[]), "of_module.py:136-146", "exec")


def module_golden(g):
    code = module_statements()
    old = ref_loader.of_library("old")
    rng = np.random.default_rng(2024)
    cases = 6
    g["module_n_cases"] = cases
    for c in range(cases):
        N = [4, 7, 30, 50, 120, 9][c]
        # centred pixel coordinates (of_module.py:96-103) or metric ones; homogeneous rows
        scale = [200.0, 150.0, 0.4, 300.0, 0.5, 100.0][c]
        x = np.ones((N, 3)); x[:, :2] = rng.uniform(-scale, scale, (N, 2))
        n = np.array([rng.normal(0, 0.05), rng.normal(0, 0.05), 1.0]); n /= np.linalg.norm(n)
        v_true = rng.uniform(-1, 1, 3)
        d_true = rng.uniform(0.5, 4.0, N)
        # translational flow of points at individual depths + noise
        u = np.zeros((N, 3))
        for i in range(N):
            X = x[i]
            u[i] = np.dot(n, X) / d_true[i] * (v_true - v_true[2] * X)
        u[:, :2] += rng.normal(0, 0.002 * scale * (c % 2), (N, 2))
        u[:, 2] = 0.0
        v_prior = v_true + rng.normal(0, 0.05, 3)
        feas, dist = old["r_tilde"](x, u, n, v_prior)
        ns = {"np": np, "feasible_new": x, "feasible_flow": u, "feasible_dist": dist, "n": n}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            exec(code, ns)
        for k, val in (("x", x), ("u", u), ("n", n), ("v_prior", v_prior), ("dist", dist), ("feas", feas),
                       ("v", ns["v_obs"]), ("res", np.asarray(ns["R"])), ("rank", ns["rank"]), ("s", ns["s"])):
            g["module%d_%s" % (c, k)] = val


def time_evolution_golden(g):
    src = open(os.path.join(REF, "numerical_simulation", "simulation.py")).read()
    tree = ast.parse(src)
    block = next(n.value.value for n in tree.body if isinstance(n, ast.Expr) and isinstance(n.value, ast.Constant)
                 and isinstance(n.value.value, str) and "# Time analysis" in n.value.value)
    text = block[block.index("# Time analysis"):]
    sub = ast.parse(text)
    keep = []
    for st in sub.body:                       # up to and including the `for i in range(k)` loop; plotting is dropped
        keep.append(st)
        if isinstance(st, ast.For):
            break
    code = compile(ast.Module(body=keep, type_ignores=[]), "simulation.py:472-499", "exec")
    sim = ref_loader.simulation()
    pts = np.loadtxt(os.path.join(REF, "numerical_simulation", "points.txt"))
    trace = {"data": [], "i": []}

    def hook(*a):
        if len(a) == 1 and isinstance(a[0], np.ndarray):
            trace["data"].append(a[0].copy())
        elif len(a) == 1:
            trace["i"].append(a[0])

    ns = dict(sim)
    ns.update(np=np, print=hook, data=pts.copy(), linear_velocity=np.array([1, 1, 1]), angular_velocity=1 * np.array([1, 1, 1]),
              height_above_gr=1, normal_vector=np.array([0, 0, 1]), translation=np.array([0.02, 0, 0.205]),
              ang_vel_sig=0.00071, translation_sig=0.005, height_sig=0.01, flow_sig=0.056 * np.sqrt(2) * 1.23,
              position_sig=0.056 * 1.23, normal_sig=0.00065)
    # of_simulation reads `iterations` and `true_flow` from ITS globals: the functions were exec'd into `sim`, and the
    # block assigns true_flow in the namespace it runs in -- run the block in that same namespace
    sim.update(ns)
    sim["iterations"] = 4
    np.random.seed(31)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        exec(code, sim)
    k = len(trace["data"])
    assert k == 100 and trace["i"] == list(range(100))
    d0 = pts.copy(); d0[:, 0] -= d0[:, 0].mean(); d0[:, 1] -= d0[:, 1].mean(); d0 *= 10
    pos = np.array([d0] + trace["data"][:-1])                 # positions at the START of every step
    g["te_pos"] = pos
    g["te_heights"] = 1.0 + np.arange(100) * 1.0              # h += v.n = 1 per step (checked against the namespace below)
    assert float(sim["height_above_gr"]) == 101.0
    g["te_final_pos"] = trace["data"][-1]
    # reference statistics at three steps, 400 trials each, through the reference's of_simulation on the traced points
    for step in (0, 7, 60):
        sim["iterations"] = 400
        h = float(g["te_heights"][step])
        sim["true_flow"] = sim["generate_test_data"](pos[step], sim["linear_velocity"], sim["angular_velocity"], h,
                                                     sim["normal_vector"], sim["translation"])
        np.random.seed(1000 + step)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            vo, _, _ = sim["of_simulation"](sim["linear_velocity"], sim["angular_velocity"], h, sim["normal_vector"],
                                            sim["translation"], pos[step], 0.00071, 0.005, 0.01, 0.056 * np.sqrt(2) * 1.23,
                                            0.056 * 1.23, 0.00065)
        g["te_ref_mean_%d" % step], g["te_ref_std_%d" % step] = vo.mean(0), vo.std(0)
    g["te_ref_trials"] = 400


def live_sorting_golden(g):
    relpath = os.path.join("numerical_simulation", "simulation.py")
    src = open(os.path.join(REF, relpath)).read()
    tree = ast.parse(src)
    sim = ref_loader.simulation()
    pts_path = os.path.join(REF, "numerical_simulation", "points.txt")
    head, live = [], []
    for n in tree.body:
        if isinstance(n, (ast.FunctionDef, ast.Import, ast.ImportFrom)):
            continue
        if isinstance(n, ast.Expr) and isinstance(n.value, ast.Constant):
            continue
        if n.lineno <= 178:
            head.append(n)
        elif 753 <= n.lineno <= 774:
            live.append(n)
    code_head = compile(ast.Module(body=head, type_ignores=[]), "simulation.py:122-178", "exec")
    code_live = compile(ast.Module(body=live, type_ignores=[]), "simulation.py:753-774", "exec")
    for tag, seed in (("a", 71), ("b", 72)):
        ns = ref_loader.simulation()            # the functions' globals ARE this dict: the statements must run in it
        real_loadtxt = np.loadtxt

        class NP(object):                       # np with loadtxt redirected to the reference directory
            def __getattr__(self, k):
                if k == "loadtxt":
                    return lambda f, *a, **kw: real_loadtxt(pts_path if f == "points.txt" else f, *a, **kw)
                return getattr(np, k)
        ns["np"] = NP()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            exec(code_head, ns)
            ns["iterations"] = 300
            np.random.seed(seed)
            exec(code_live, ns)
        if tag == "a":
            g["live_data"], g["live_true_flow"] = np.array(ns["data"]), np.array(ns["true_flow"])
            g["live_velocity"], g["live_height"] = np.array(ns["linear_velocity"], dtype=np.float64), float(ns["height_above_gr"])
            g["live_minang"] = float(ns["minang"])          # Python 3 here: 10/360*2*pi = 0.1745 (0 under Python 2)
            g["live_seed"] = seed
            # the rotation angles the live section drew (first draws of the seeded legacy stream)
            st = np.random.RandomState(seed)
            nsec = 2 * int(200 / 3) - int(200 / 5)
            g["live_angles"] = np.array([st.uniform(ns["minang"], 2 * np.pi - ns["minang"]) for _ in range(nsec)])
        for name in ("backward_para", "backward_dist", "forward_para", "forward_dist", "backward_res", "forward_res"):
            g["live_%s_%s" % (name, tag)] = np.array(ns[name])
    g["live_iterations"] = 300


if __name__ == "__main__":
    if not ref_loader.available():
        sys.exit(ref_loader.MISSING)
    g = {}
    module_golden(g)
    time_evolution_golden(g)
    live_sorting_golden(g)
    np.savez_compressed(os.path.join(OUT, "velocity_golden_r2.npz"), **g)
    print(os.path.getsize(os.path.join(OUT, "velocity_golden_r2.npz")), "bytes,", len(g), "arrays")
