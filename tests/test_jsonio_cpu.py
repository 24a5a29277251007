"""The reference's JSON problem format (default/json.rs:11-95): round trip through clarabel.rs_b200/jsonio.py and its
own examples/data/hs35.json, stored verbatim as tests/golden/reference_data/hs35.json.  CPU only."""
import importlib.util
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp

import clarabel_rs_b200 as cb
import oracle
import ref_problems as rp

_spec = importlib.util.spec_from_file_location("jsonio", os.path.join(os.path.dirname(cb.pkg.__file__), "jsonio.py"))
jsonio = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(jsonio)


def test_round_trip_all_cone_kinds(tmp_path):
    rng = np.random.default_rng(0)
    cones = [("zero", 2), ("nonneg", 3), ("soc", 4), ("psd", 2), ("exp", 3), ("pow", 0.3), ("genpow", ([0.5, 0.5], 2))]
    m, n = 2 + 3 + 4 + 3 + 3 + 3 + 4, 5
    P = sp.random(n, n, density=0.5, random_state=1); P = (P + P.T + sp.identity(n)).tocsc()
    A = sp.random(m, n, density=0.4, random_state=2, format="csc")
    q, b = rng.standard_normal(n), rng.standard_normal(m)
    path = tmp_path / "p.json"
    jsonio.save_problem(path, P, q, A, b, cones, settings={"max_iter": 50, "time_limit": float("inf"), "tol_feas": 1e-7})
    d = jsonio.load_problem(path)
    assert (d["P"] != sp.triu(P)).nnz == 0 and (d["A"] != A).nnz == 0
    assert np.array_equal(d["q"], q) and np.array_equal(d["b"], b)
    assert d["cones"] == cones
    assert d["settings"] == {"max_iter": 50, "time_limit": float("inf"), "tol_feas": 1e-7}
    raw = json.loads(path.read_text())
    assert raw["cones"][0] == {"ZeroConeT": 2} and raw["cones"][4] == {"ExponentialConeT": []} and raw["cones"][5] == {"PowerConeT": 0.3} and raw["cones"][6] == {"GenPowerConeT": [[0.5, 0.5], 2]}


def test_rejects_unknown_cones(tmp_path):
    base = {"P": {"m": 1, "n": 1, "colptr": [0, 0], "rowval": [], "nzval": []}, "q": [0.0],
            "A": {"m": 3, "n": 1, "colptr": [0, 0], "rowval": [], "nzval": []}, "b": [0.0, 0.0, 0.0]}
    for cone in ({"FancyConeT": 3},):
        p = tmp_path / "bad.json"
        p.write_text(json.dumps(dict(base, cones=[cone])))
        with pytest.raises(ValueError):
            jsonio.load_problem(p)


def test_reference_data_file_hs35():
    d = jsonio.load_problem(os.path.join(os.path.dirname(__file__), "golden", "reference_data", "hs35.json"))
    P, q, A, b, cones = rp.hs35()
    assert (d["P"] != P).nnz == 0 and (d["A"] != A).nnz == 0 and list(d["q"]) == q and list(d["b"]) == b
    assert d["cones"] == cones
    assert d["settings"]["max_iter"] == 200 and d["settings"]["time_limit"] == float("inf")
    ipm = oracle.IPM(d["P"], d["q"], d["A"], d["b"], d["cones"],
                     settings=oracle.default_settings(**{k: v for k, v in d["settings"].items()}))
    ipm.set_perm(np.arange(ipm.N))
    r = ipm.solve()
    assert r["status"] == "Solved" and np.linalg.norm(r["x"] - [4 / 3, 7 / 9, 4 / 9]) <= 1e-6
