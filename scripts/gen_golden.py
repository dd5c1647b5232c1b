#!/usr/bin/env python
"""Generates tests/golden/*.json from the REFERENCE ITSELF, run in this container.

  parser_golden.json   every dataset MPS file parsed by the reference's libmps_parser (free AND fixed mode):
                       either the error flag or a digest + the full arrays for small files
  simplex_golden.json  optimal objectives from the reference's CPU dual simplex (cpp/src/dual_simplex)
  reference_pins.json  known answers copied from the reference's own tests (with file:line provenance)

Needs /root/reference and oracle/_ref (make -C oracle ref).  The outputs are committed; the GPU box never runs this.
"""
from __future__ import annotations

import glob
import gzip
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_cpu  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
MPS = os.path.join(GOLD, "mps")


def digest(arr) -> str:
    a = np.ascontiguousarray(arr)
    return hashlib.sha256(a.tobytes()).hexdigest()[:16]


def model_record(m: ref_cpu.MpsModel, full: bool) -> dict:
    rec = dict(m=m.m, n=m.n, nnz=m.nnz, maximize=m.maximize, objective_offset=m.objective_offset,
               objective_scaling_factor=m.objective_scaling_factor, problem_name=m.problem_name,
               objective_name=m.objective_name,
               digests=dict(offsets=digest(m.offsets), indices=digest(m.indices), values=digest(m.values),
                            rhs=digest(m.rhs), c=digest(m.c), var_lb=digest(m.var_lb), var_ub=digest(m.var_ub),
                            con_lb=digest(m.con_lb), con_ub=digest(m.con_ub)),
               var_types=m.var_types.decode(errors="replace").replace("\x00", "C"),
               n_row_types=len(m.row_types))
    if full:
        f = lambda a: [None if not np.isfinite(v) else float(v) for v in a]  # noqa: E731
        inf = lambda a: [("inf" if v > 0 else "-inf") if np.isinf(v) else float(v) for v in a]  # noqa: E731
        rec["arrays"] = dict(offsets=m.offsets.tolist(), indices=m.indices.tolist(), values=f(m.values),
                             rhs=f(m.rhs), c=f(m.c), var_lb=inf(m.var_lb), var_ub=inf(m.var_ub),
                             con_lb=inf(m.con_lb), con_ub=inf(m.con_ub))
        rec["var_names"] = m.var_names
        rec["row_names"] = m.row_names
    return rec


def mps_files():
    out = []
    for sub in ("linear_programming", "mip"):
        for p in sorted(glob.glob(os.path.join(MPS, sub, "*.mps*"))):
            out.append(p)
    return out


def materialise(path: str) -> str:
    if path.endswith(".gz"):
        tmp = tempfile.NamedTemporaryFile(suffix=".mps", delete=False)
        tmp.write(gzip.open(path).read())
        tmp.close()
        return tmp.name
    return path


def main():
    parser = {}
    simplex = {}
    for path in mps_files():
        key = os.path.relpath(path, MPS).replace(".gz", "")
        real = materialise(path)
        entry = {}
        for mode, fixed in (("free", False), ("fixed", True)):
            try:
                m = ref_cpu.parse_mps(real, fixed_format=fixed)
                entry[mode] = dict(ok=True, **model_record(m, full=m.nnz <= 200))
            except ValueError as e:
                entry[mode] = dict(ok=False, error=str(e)[:200])
        parser[key] = entry
        if entry["free"]["ok"] and entry["free"]["m"] > 0 and entry["free"]["nnz"] > 0:
            try:
                r = ref_cpu.dual_simplex_mps(real, time_limit=600.0)
                simplex[key] = dict(status=r["status"], objective=r["objective"], iterations=r["iterations"],
                                    seconds=round(r["seconds"], 4))
                print(key, simplex[key], flush=True)
            except Exception as e:  # noqa: BLE001
                simplex[key] = dict(status="EXCEPTION", error=str(e)[:200])
    json.dump(parser, open(os.path.join(GOLD, "parser_golden.json"), "w"), indent=1, sort_keys=True)
    json.dump(simplex, open(os.path.join(GOLD, "simplex_golden.json"), "w"), indent=1, sort_keys=True)

    pins = {
        "_provenance": "values copied from the reference's own test sources; paths relative to /root/reference",
        "afiro_objective": dict(value=-464.7531, rel=1e-6,
                                source="python/cuopt/cuopt/tests/linear_programming/test_lp_solver.py:101-121,592-606"),
        "afiro_objective_cpp": dict(value=-464.0, rel=1e-2, source="cpp/tests/linear_programming/pdlp_test.cu:58-84"),
        "afiro_methodical1_initial_step_size": dict(value=1.4893, abs=1e-4,
                                                    source="cpp/tests/linear_programming/pdlp_test.cu:237-283"),
        "afiro_methodical1_initial_primal_weight": dict(value=0.0141652, abs=1e-4,
                                                        source="cpp/tests/linear_programming/pdlp_test.cu:237-283"),
        "afiro_default_primal": dict(
            rel=1e-4, source="python/cuopt/cuopt/tests/linear_programming/test_lp_solver.py:430-476",
            settings="defaults (tolerances 1e-4, Stable2), method PDLP",
            values={"X01": 80.00603991232295, "X02": 25.52673622717911, "X03": 54.498387438550935, "X04": 0.0,
                    "X06": 73.04802363832049, "X07": 0.0, "X08": 0.0, "X09": 0.0, "X10": 0.0, "X11": 0.0,
                    "X12": 0.0, "X13": 0.0, "X14": 18.232656093528156, "X15": 0.0, "X16": 0.0,
                    "X22": 499.9879512761402, "X23": 475.85273137206457, "X24": 24.097841116452646, "X25": 0.0,
                    "X26": 0.0, "X28": 0.0, "X29": 0.0, "X30": 0.0, "X31": 0.0, "X32": 0.0, "X33": 0.0, "X34": 0.0,
                    "X35": 0.0, "X36": 339.88604763129206, "X37": 25.615058891374325, "X38": 0.0, "X39": 0.0}),
        "good_max_objective": dict(value=17.0, abs=1e-4, source="cpp/tests/linear_programming/pdlp_test.cu:909-925"),
        "max_offset_objective": dict(value=0.0, abs=1e-4, source="cpp/tests/linear_programming/pdlp_test.cu:927-943"),
        "c_api_ranged_objective": dict(
            value=32.0, abs=1e-3, source="cpp/tests/linear_programming/c_api_tests/c_api_test.c:761-874"),
    }
    json.dump(pins, open(os.path.join(GOLD, "reference_pins.json"), "w"), indent=1)
    writer_golden()


def writer_golden():
    """writer_golden.json: the reference parser's reading of the MPS file this repo's writer writes for the LP of
    tests/test_file_writers.py (needs cuopt_b200/lib/libcuopt.so too; the file is written before any GPU work)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cuopt_b200 import capi, lpgen
    from test_file_writers import WRITER_LP, lp_digests, write_via_solve
    lp = lpgen.sparse_lp(WRITER_LP["m"], WRITER_LP["n"], WRITER_LP["nnz_per_row"], seed=WRITER_LP["seed"])
    p = capi.Problem.create_ranged(lp.offsets, lp.indices, lp.values, lp.con_lb, lp.con_ub, lp.c, lp.var_lb, lp.var_ub)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "written.mps")
        write_via_solve(p, path)
        m = ref_cpu.parse_mps(path)
        with open(path, "rb") as f:
            sha = hashlib.sha256(f.read()).hexdigest()
    rec = dict(lp=f"lpgen.sparse_lp({WRITER_LP['m']}, {WRITER_LP['n']}, {WRITER_LP['nnz_per_row']}, "
                  f"seed={WRITER_LP['seed']})", file_sha256=sha,
               reference_parse=dict(m=m.m, n=m.n, digests=lp_digests(m.m, m.n, m.offsets, m.indices, m.values, m.c,
                                                                     m.con_lb, m.con_ub, m.var_lb, m.var_ub)))
    with open(os.path.join(GOLD, "writer_golden.json"), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if sys.argv[1:] == ["writer"]:
        writer_golden()
    else:
        main()
