"""The arctangent constants of csrc/d2dx_math.cuh are the ones scripts/atan_table.py derives, and their truncation bound holds."""
import importlib.util
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MATH = os.path.join(ROOT, "drone-sim-python_b200", "csrc", "d2dx_math.cuh")


def _script():
    spec = importlib.util.spec_from_file_location("atan_table", os.path.join(ROOT, "scripts", "atan_table.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _doubles(text):
    return [float(v) for v in re.findall(r"[-+]?\d+\.\d*(?:e[-+]?\d+)?", text)]


def test_truncation_bound_in_exact_arithmetic():
    mod = _script()
    p, _ = mod.coefficients()
    assert mod.check([float(c) for c in p]) < mod.BOUND


def test_header_constants_match_the_script():
    mod = _script()
    src = open(MATH).read()
    tab = _doubles(re.search(r"kAtanTab\[kAtanTabLen\] = \{(.*?)\};", src, re.S).group(1))
    assert tab == mod.table()
    # atan core: kTab[20..23] hold -P, highest power first
    body = re.search(r"kTab\[56\] = \{(.*?)\};", src, re.S).group(1)
    core = [v for k in (20, 22) for v in _doubles(re.search(r"/\*%d\*/([^/]*)" % k, body).group(1))]
    p, _ = mod.coefficients()
    assert core == [-float(c) for c in reversed(p)]
