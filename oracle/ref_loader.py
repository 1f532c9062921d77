"""Loads the REFERENCE's own functions (verbatim, at run time) for pinning the oracle.

Test infrastructure only. Works only where OFB_REFERENCE_DIR names a checkout of the original
Python project. The repository does not carry it: without it the live comparisons skip and the
committed golden outputs under tests/golden/ pin the oracle. simulation.py /
velocity_measurment_node / evaluate_exp.py cannot be imported (matplotlib / rospy missing, sweeps
run at import), so their FunctionDefs are AST-extracted and exec'd in a namespace holding numpy.
Nothing is copied into the repo.
"""
import ast
import os

import numpy as np

REF = os.environ.get("OFB_REFERENCE_DIR", "")
MISSING = "needs OFB_REFERENCE_DIR (a checkout of the original project)"


def available():
    return bool(REF) and os.path.isfile(os.path.join(REF, "numerical_simulation", "simulation.py"))


def load_functions(relpath, names=None, extra_globals=None):
    src = open(os.path.join(REF, relpath)).read()
    tree = ast.parse(src)
    ns = {"np": np, "__builtins__": __builtins__}
    if extra_globals:
        ns.update(extra_globals)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and (names is None or node.name in names):
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, relpath, "exec"), ns)
    return ns


def simulation():
    return load_functions("numerical_simulation/simulation.py",
                          ["generate_test_data", "solve_lgs", "of_simulation", "feas_simulation",
                           "feasibility", "overlap"])


def node():
    return load_functions("velocity_measurment_node", ["generate_test_data", "solve_lgs"])


def evaluate_exp():
    return load_functions("flight_experiments/evaluate_exp.py", ["solve_lgs"])


def of_library(which="root"):
    rel = {"root": "of_library.py",
           "old": "sensor_precision_experiments/pixhawk_pure_IMU/of_library.py"}[which]
    return load_functions(rel, ["pix_trans", "r_tilde", "static_immobile"])
