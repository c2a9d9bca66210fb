"""bench.py must print its headline line even when one of the extra configurations (other_configs) fails: each
is guarded and its failure becomes that configuration's record.  No GPU needed: the contexts are made to fail."""
import importlib.util
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    spec = importlib.util.spec_from_file_location("_bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_default_extras_depend_on_world_size(monkeypatch):
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    assert bench.parse().extra == "c2f,c2m,w,c3,c4,c5,c4o"
    monkeypatch.setenv("WORLD_SIZE", "8")
    assert bench.parse().extra == "c5"           # the configuration BASELINE.json names for 8 GPUs
    monkeypatch.setattr(sys, "argv", ["bench.py", "--extra", ""])
    assert bench.parse().extra == ""


def test_failing_extra_config_becomes_a_record(monkeypatch, capsys):
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    a = bench.parse()
    closed = []

    class Boom(RuntimeError):
        pass

    class FakeCtx:
        def __init__(self, *args, **kw):
            pass

        def close(self):
            closed.append(1)

        def add_space(self, *args, **kw):
            raise Boom("no device")

    def fail(*args, **kw):
        raise Boom("no device")

    fake = types.SimpleNamespace(
        _lib=types.SimpleNamespace(load=lambda: types.SimpleNamespace()),
        B200Context=FakeCtx,
        B200CSR=types.SimpleNamespace(stencil_free=fail, stencil=fail),
        cgs2=None, mgs2=None, cgs=None, mgs=None, mgs2b=None)
    # the legs that use the real package fail too, also where a GPU is present: tools/run_configs.py (in this
    # process) cannot create a context, and the c4o child process sees no CUDA device
    import krylovkit_jl_b200 as kk
    monkeypatch.setattr(kk, "B200Context", fail)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    out = bench.other_configs(fake, a, 0, 1, 0, None)
    assert set(out) == {"c2_matrix_free", "c2_reference_default_orth", "widened_solvers", "c3", "c4", "c5", "c4_onepass"}
    for name, rec in out.items():
        assert rec["ok"] is False
        if name in ("widened_solvers", "c4_onepass"):   # tools/run_configs.py on the real package / bench.py's child
            assert "B200Error" in rec["error"] or "Boom" in rec["error"] or "CUDA" in rec["error"]   # process: "no CUDA device"
        else:
            assert "Boom: no device" in rec["error"]
    assert len(closed) == 5                     # every failed in-process configuration gave its context back
    assert "Boom" in capsys.readouterr().err    # the traceback goes to stderr, the JSON line stays clean


def test_reference_default_orth_extra_runs_on_the_simulator(monkeypatch):
    """The success path of an extra configuration — bench.other_configs 'c2m' (literal MGS2 and the flagged blocked
    form on the headline operator, parity against a committed oracle result) — on tests/hostsim.py at a small size,
    with a golden record made by the oracle on the spot.  Also proves the slab column budget of that block."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostsim
    import krylovkit_jl_b200 as kk
    from oracle import krylov_oracle as ko
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--nx", "30", "--ny", "22", "--krylovdim", "12", "--cycles", "3",
                                      "--extra", "c2m"])
    a = bench.parse()
    A, x0 = ko.stencil_matrix(30, 22), ko.splitmix_vector(bench.SEED, 660)
    ov, _, oi = ko.eigsolve_lanczos(A, x0, 4, "SR", krylovdim=12, maxiter=2, tol=0.0, orth=ko.Orth(ko.MGS2))
    fake = {"c2_mgs2": {"grid": [30, 22, 1], "krylovdim": 12,
                        "after_cycles": {"2": {"ritz": [float(v) for v in ov[:4]], "numops": oi["numops"]}}}}
    monkeypatch.setattr(bench.json, "load", lambda f: fake)
    with hostsim.installed(fused=True):
        out = bench.other_configs(kk, a, 0, 1, 0, None)
    rec = out["c2_reference_default_orth"]
    assert "error" not in rec, rec
    for name in ("mgs2_reference_default", "mgs2_blocked_flagged"):
        assert rec[name]["numops"] == 12 + 2 * (12 - (3 * 12) // 5) and rec[name]["value"] > 0
        assert rec[name]["parity"]["ok"] and rec[name]["parity"]["numops"] == oi["numops"]


def test_widened_solver_records_run_on_the_simulator():
    """What bench.other_configs 'w' calls — tools/run_configs.py cg() and widened(lsmr=False), loaded by path — on
    tests/hostsim.py at a small size: every record is produced and carries its residual identity."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostsim
    spec = importlib.util.spec_from_file_location("_rc_under_test", os.path.join(ROOT, "tools", "run_configs.py"))
    rc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rc)
    with hostsim.installed(fused=True):
        cg = rc.cg(40, 30)
        rec = rc.widened(40, 30, lsmr=False)
    assert set(cg) == {"chained_32", "fused_step", "literal_mirror"}
    for r in cg.values():
        assert r["numiter"] == 200 and r["||A x + r - b||/||b||"] < 1e-12
    assert set(rec) == {"bicgstab", "arnoldi_eigsolve", "blocklanczos_p4", "blocklanczos_p4_fast_block", "exponentiate"}
    assert rec["bicgstab"]["||A x - b||/||b||"] < 1e-10 and rec["exponentiate"]["converged"] == 1
    assert rec["blocklanczos_p4"]["numops"] == rec["blocklanczos_p4_fast_block"]["numops"]
    assert abs(rec["blocklanczos_p4"]["ritz"][0] - rec["blocklanczos_p4_fast_block"]["ritz"][0]) < 1e-10


def test_onepass_extra_runs_on_the_simulator(monkeypatch):
    """The success path of bench.other_configs 'c4o' (config 4, two-pass reference step against the flagged one-pass
    step, run last) on tests/hostsim.py at 20 000 rows: every record is produced, the singular values of the two modes
    agree within the Float32 bar, the one-pass mode streams fewer passes; also proves the column budgets of that block."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostsim
    import krylovkit_jl_b200 as kk
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--extra", "c4o", "--c4-rows", "20000"])
    monkeypatch.setenv("B2K_BENCH_CHILD", "1")          # the in-process body (bench.py runs it in a child process)
    a = bench.parse()
    with hostsim.installed(fused=True):
        out = bench.other_configs(kk, a, 0, 1, 0, None)
    rec = out["c4_onepass"]
    assert "error" not in rec, rec
    for oname in ("mgs2", "cgsr_eta0.75"):
        two, one = rec[f"{oname}:two_pass_reference"], rec[f"{oname}:one_pass_flagged"]
        assert two["converged"] >= 6 and one["converged"] >= 6 and one["ok"]
        assert two["passes_over_A"] == two["numops"] and one["passes_over_A"] < one["numops"]
        assert one["max_rel_diff_sigma_vs_two_pass"] <= 3e-5


def test_onepass_extra_is_isolated_in_a_child_process(monkeypatch):
    """bench.other_configs 'c4o' without B2K_BENCH_CHILD spawns `bench.py --extra c4o` as a child and turns whatever
    happens there into a record: here (the child sees no CUDA device) the child's context creation fails, the child
    still prints its record, and the parent carries it — the parent itself never touches the one-pass kernel."""
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--extra", "c4o", "--c4-rows", "4000"])
    monkeypatch.delenv("B2K_BENCH_CHILD", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    a = bench.parse()
    out = bench.other_configs(types.SimpleNamespace(_lib=types.SimpleNamespace(load=lambda: None)), a, 0, 1, 0, None)
    rec = out["c4_onepass"]
    assert rec["ok"] is False and "error" in rec and ("B200Error" in rec["error"] or "CUDA" in rec["error"] or "cuda" in rec["error"])


def test_headline_path_runs_on_the_simulator_and_prints_the_contract(monkeypatch, capsys, tmp_path):
    """bench.run_ours end to end on tests/hostsim.py at a small size — the resident job, the host-buffer (e2e) leg with
    its pinned buffers, the per-kernel profile and the assembly of the one JSON line — so that the host code of the
    headline is exercised on a box without a GPU.  The line must parse STRICTLY (no NaN / Infinity tokens) and carry
    the keys of the bench contract; the Ritz values of both legs must agree with the oracle on the same (A, x0).
    --dump-outputs (with fewer sampled rows than n) writes what the last timed job returned: float64 arrays that agree
    with the oracle's values, vectors and residuals at the sampled rows."""
    import json
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostsim
    from oracle import krylov_oracle as ko
    bench = _load_bench()
    dump = tmp_path / "outputs"
    monkeypatch.setattr(bench, "DUMP_ROWS", 500)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--nx", "40", "--ny", "30", "--krylovdim", "12", "--cycles", "3", "--steps", "2",
                                      "--warmup", "1", "--no-cpu-baseline", "--extra", "", "--dump-outputs", str(dump)])
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("B2K_BENCH_CHILD", raising=False)
    a = bench.parse()
    with hostsim.installed(fused=True):
        bench.run_ours(a)
    out = capsys.readouterr().out.strip().splitlines()
    assert len(out) == 1                                         # ONE line

    def no_constants(tok):
        raise AssertionError(f"non-standard JSON token {tok}")
    line = json.loads(out[0], parse_constant=no_constants)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["dtype"] == "f64" and line["gpu_launches"] > 0
    assert line["numops_per_step"] == 12 + 2 * (12 - (3 * 12) // 5) and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0 and line["e2e"]["value"] > 0
    ov, ovecs, oi = ko.eigsolve_lanczos(ko.stencil_matrix(40, 30), ko.splitmix_vector(bench.SEED, 1200), 4, "SR", krylovdim=12,
                                        maxiter=3, tol=0.0, orth=ko.Orth(ko.CGS2))
    assert oi["numops"] == line["numops_per_step"]
    assert max(abs(x - y) for x, y in zip(line["ritz_values"], ov[:4])) < 1e-10
    got = {p.stem: np.load(p) for p in dump.iterdir()}
    assert set(got) == {"ritz_values", "ritz_vectors", "residuals", "normres", "counts", "sample_rows"}
    assert all(x.dtype == np.float64 for x in got.values())
    rows = got["sample_rows"].astype(np.int64)
    assert len(rows) == 500 and np.all(np.diff(rows) > 0) and rows[-1] < 1200
    assert got["ritz_values"].tolist() == line["ritz_values"]
    assert got["counts"].tolist() == [oi["converged"], oi["numiter"], oi["numops"]]
    np.testing.assert_allclose(got["normres"], oi["normres"][:4], rtol=1e-8, atol=1e-14)
    np.testing.assert_allclose(got["ritz_vectors"], np.stack([v[rows] for v in ovecs[:4]]), atol=1e-10)
    np.testing.assert_allclose(got["residuals"], np.stack([r[rows] for r in oi["residual"][:4]]), atol=1e-10)


def test_json_safe_makes_any_record_strictly_parseable():
    import json
    import numpy as np
    bench = _load_bench()
    rec = {"a": float("nan"), "b": [np.float32(1.5), np.inf, {"c": np.int64(3), "d": np.bool_(True)}], "e": np.array([1.0, np.nan])}
    txt = json.dumps(bench.json_safe(rec), allow_nan=False, default=str)
    assert json.loads(txt) == {"a": "nan", "b": [1.5, "inf", {"c": 3, "d": True}], "e": [1.0, "nan"]}


def test_config4_extra_runs_on_the_simulator_with_the_truth_check(monkeypatch):
    """bench.other_configs 'c4' (two-pass GKL, three orthogonalizers) on the simulator at 4000 rows, once without a
    committed truth for that shape and once with one: the record gains the distance from the truth and its verdict."""
    import json
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostsim
    import krylovkit_jl_b200 as kk
    bench = _load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--extra", "c4", "--c4-rows", "4000"])
    a = bench.parse()
    with hostsim.installed(fused=True):
        rec = bench.other_configs(kk, a, 0, 1, 0, None)["c4"]
    assert "error" not in rec and "max_rel_err_sigma_vs_float64_truth" not in rec["mgs2_reference_default"]
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "fullsize.json")))
    gold["c4_truth"] = {"shape": [4000, 512], "sigma_float64_truth": rec["mgs2_reference_default"]["sigma"]}
    monkeypatch.setattr(bench.json, "load", lambda f: gold)
    with hostsim.installed(fused=True):
        rec = bench.other_configs(kk, a, 0, 1, 0, None)["c4"]
    assert rec["cgsr_eta0.75"]["ok"] and rec["cgsr_eta0.75"]["max_rel_err_sigma_vs_float64_truth"] < 3e-5
