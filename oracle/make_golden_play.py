#!/usr/bin/env python
"""TEST INFRASTRUCTURE (not product code).  Freezes known answers of the reference play script's pure helper functions
(`_quantize_xy`, `_hash_obstacles_xy`, `_bootstrap_mean_ci`, `_infer_done_reason`, `_apply_mass_mode_to_obs`;
OIGE/scripts/rlgames_play_loopz.py:135-171,493-533,560-621)
into tests/golden/play_metrics.json.  The script itself imports hydra / Isaac Sim at module level, so the function definitions are
taken out of its syntax tree and executed unmodified.  Needs a reference checkout:
USV_REFERENCE_ROOT=<reference checkout> python oracle/make_golden_play.py"""
import ast
import hashlib
import json
import math
import os
from typing import Any, Dict, Optional, Tuple

import numpy as np

REF = os.path.join(os.environ.get("USV_REFERENCE_ROOT", ""), "omniisaacgymenvs", "scripts", "rlgames_play_loopz.py")
WANT = {"_quantize_xy", "_hash_obstacles_xy", "_bootstrap_mean_ci", "_infer_done_reason", "_apply_mass_mode_to_obs"}


def load():
    src = open(REF).read()
    tree = ast.parse(src)
    ns = dict(np=np, hashlib=hashlib, math=math, Any=Any, Dict=Dict, Optional=Optional, Tuple=Tuple)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in WANT:
            exec(compile(ast.Module([node], []), REF, "exec"), ns)
    return ns


def main():
    ns = load()
    rng = np.random.default_rng(7)
    layouts = []
    for k in range(6):
        xy = (rng.random((16, 2)) * 24 - 12).astype(np.float32)
        if k % 2:
            xy[rng.integers(0, 16, size=3)] = 999.0            # limbo obstacles
        if k == 4:
            xy = np.round(xy * 200) / 200                      # values on quantisation half-steps (round half to even)
        layouts.append({"xy": xy.tolist(), "quant": ns["_quantize_xy"](xy, quant_m=0.01).tolist(),
                        "hash": ns["_hash_obstacles_xy"](xy, quant_m=0.01),
                        "hash_shuffled": ns["_hash_obstacles_xy"](xy[rng.permutation(16)], quant_m=0.01),
                        "hash_q05": ns["_hash_obstacles_xy"](xy, quant_m=0.05)})
    boots = []
    for k, n in enumerate((1, 2, 17, 200)):
        v = rng.normal(size=n) * (k + 1)
        if n > 2:
            v[::5] = np.nan
        boots.append({"values": [None if np.isnan(x) else float(x) for x in v],
                      "ci": list(ns["_bootstrap_mean_ci"](v, rng=np.random.default_rng(3)))})
    reasons = []
    for c in (0.0, 1.0):
        for o in (0.0, 1.0):
            for g in (0.0, 1.0):
                reasons.append({"collision": c, "out_of_bounds": o, "in_goal_tolerance": g,
                                "reason": ns["_infer_done_reason"]({"collision": c, "out_of_bounds": o, "in_goal_tolerance": g})})
    mass_modes = []
    for n in (1, 2, 7, 12):
        obs = rng.normal(size=(n, 9)).astype(np.float32)
        for mode in ("normal", "zero", "shuffle", "swap", "Swap ", "bogus"):
            mass_modes.append({"obs": obs.tolist(), "mode": mode, "seed": 5,
                               "out": ns["_apply_mass_mode_to_obs"](obs, mode=mode, rng=np.random.default_rng(5), warn_once={}).tolist()})
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "play_metrics.json")
    json.dump({"layouts": layouts, "bootstrap": boots, "reasons": reasons, "mass_modes": mass_modes}, open(out, "w"))
    print("wrote", os.path.normpath(out))


if __name__ == "__main__":
    main()
