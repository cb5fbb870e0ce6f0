"""CPU-side checks: the C-ABI library loads and exports every symbol include/b200adj.h declares (no compute calls
without a GPU), the product path fails loudly without a device, and the host layer mirrors the reference's plugin
surface (names, defaults, error behaviour)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import scimlsensitivity_jl_b200 as b
from scimlsensitivity_jl_b200 import _lib
from scimlsensitivity_jl_b200.problems import saveat_to_times

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    import torch
    return torch.cuda.is_available()


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "b200adj.h")).read()
    declared = set(re.findall(r"\b(b200adj_[a-z_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.b200adj_version() >= 0x000100


def test_cfg_struct_layout_matches_header():
    """The ctypes mirror must have the C struct's size: 8-byte alignment, 4 x int32 at the end."""
    hdr = open(os.path.join(ROOT, "include", "b200adj.h")).read()
    body = hdr[hdr.index("typedef struct b200adj_cfg {"):hdr.index("} b200adj_cfg;")]
    names = re.findall(r"(\w+)\s*(?:,|;)", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    fields = [n for n, _ in _lib.Cfg._fields_]
    assert [n for n in names if n in fields] == fields
    assert C.sizeof(_lib.Cfg) == _lib.load().b200adj_sizeof_cfg() == 176


@pytest.mark.skipif(_has_gpu(), reason="checks the no-device behaviour")
def test_no_cpu_fallback_without_device():
    with pytest.raises(b.B200AdjError) as ei:
        b.DeviceEnsemble("lorenz", "gauss", "tsit5_fixed", 8, np.linspace(0, 1, 11), (0.0, 1.0), 0.01)
    assert ei.value.code == -3 and "no CPU fallback" in str(ei.value)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "scimlsensitivity.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in txt and "adjoint_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f


def test_sensealg_structs_mirror_reference_defaults():
    # src/sensitivity_algorithms.jl:254-278, 378-405, 486-510, 591-611
    assert b.BacksolveAdjoint().checkpointing is True and b.BacksolveAdjoint().noisemixing is False
    assert b.InterpolatingAdjoint().checkpointing is False
    q = b.QuadratureAdjoint()
    assert (q.abstol, q.reltol) == (1e-6, 1e-3)
    assert b.GaussAdjoint().checkpointing is False
    # GaussKronrodAdjoint (:689-703) belongs to AbstractGAdjoint (:712) and shares its traits (:1675-1699)
    assert b.GaussKronrodAdjoint().checkpointing is False and b.supports_functor_params(b.GaussKronrodAdjoint())
    assert b.sensealg_name(b.B200Adjoint(b.GaussKronrodAdjoint())) == "gauss_kronrod"
    for A in (b.BacksolveAdjoint, b.InterpolatingAdjoint, b.QuadratureAdjoint, b.GaussAdjoint, b.GaussKronrodAdjoint):
        a = A()
        assert a.autojacvec is None and b.get_chunksize(a) == 0 and b.alg_autodiff(a) is True and b.diff_type(a) == "central"
        a2 = b.setvjp(a, b.ReverseDiffVJP(True))
        assert a2.autojacvec == b.ReverseDiffVJP(True) and type(a2) is A and b.get_jacvec(a2) is True
    w = b.B200Adjoint(b.GaussAdjoint())
    assert b.setvjp(w, b.B200VJP()).inner.autojacvec == b.B200VJP()
    assert b.ischeckpointing(b.BacksolveAdjoint()) and not b.ischeckpointing(b.InterpolatingAdjoint())
    assert b.isnoisemixing(b.BacksolveAdjoint(noisemixing=True))
    with pytest.raises(TypeError):
        b.B200Adjoint(inner="nope")


def test_saveat_semantics():
    # saveat::Number -> t0:saveat:t1 (+ end point) src/concrete_solve.jl:718-725
    ts = saveat_to_times(0.1, (0.0, 10.0))
    assert len(ts) == 101 and ts[0] == 0.0 and ts[-1] == 10.0
    ts = saveat_to_times(0.3, (0.0, 1.0))
    assert np.allclose(ts, [0.0, 0.3, 0.6, 0.9, 1.0])
    assert np.array_equal(saveat_to_times([0.5, 0.1, 0.3], (0.0, 1.0)), [0.1, 0.3, 0.5])     # sorted (:752-756)


def test_parameter_compatibility_errors():
    # src/sensitivity_interface.jl:25-29 / src/concrete_solve.jl:544-549
    prob = b.EnsembleProblem(b.ODEProblem("lorenz", [1.0, 0, 0], (0.0, 1.0), np.array([10, 28, 3])), u0s=np.ones((3, 4)))
    with pytest.raises(b.AdjointSensitivityParameterCompatibilityError):
        b.solve(prob, b.Tsit5(dt=0.01), saveat=0.1)
    prob = b.EnsembleProblem(b.ODEProblem("lorenz", [1.0, 0, 0], (0.0, 1.0), None), u0s=np.ones((3, 4)))
    with pytest.raises(ValueError):
        b.solve(prob, b.Tsit5(dt=0.01), saveat=0.1)
    prob = b.EnsembleProblem(b.ODEProblem("lorenz", [1.0, 0, 0], (0.0, 1.0), np.ones(3), callback=object()), u0s=np.ones((3, 4)))
    with pytest.raises(NotImplementedError):
        b.solve(prob, b.Tsit5(dt=0.01), saveat=0.1)
    assert b.Tsit5(adaptive=True).code == "tsit5_adaptive" and b.Tsit5(dt=0.1).code == "tsit5_fixed"
    prob = b.EnsembleProblem(b.ODEProblem("lorenz", [1.0, 0, 0], (0.0, 1.0), np.ones(3)), u0s=np.ones((3, 4)))
    with pytest.raises(ValueError):
        b.solve(prob, b.Tsit5(adaptive=True))              # adaptive solves need explicit save times
    with pytest.raises(KeyError):
        b.solve(b.EnsembleProblem(b.ODEProblem("nope", [1.0], (0.0, 1.0), np.ones(3)), u0s=np.ones((1, 4))), b.Tsit5(dt=0.01), saveat=0.1)


def test_shard_bounds_partition():
    N = 65537
    for G in (1, 2, 3, 8):
        b_ = [b.shard_bounds(N, g, G) for g in range(G)]
        assert b_[0][0] == 0 and b_[-1][1] == N and all(b_[i][1] == b_[i + 1][0] for i in range(G - 1))
        assert max(h - l for l, h in b_) - min(h - l for l, h in b_) <= 1


def test_preset_time_callback_tables_and_host_side_rejections():
    """PresetTimeCallback(tstops, AffineAffect): event tables sorted by time, one affect per time or one for all, optional
    parameter affect; everything else is refused on the host before any device call (SURVEY.md App. E)."""
    cb = b.PresetTimeCallback([8.0, 2.03, 4.0], [b.AffineAffect([1, 1], [3.0, 0]), b.AffineAffect([1, 1], [1.0, 0]), b.AffineAffect([0, 1], [2.0, 0])])
    t, sc, sh = cb.tables(2, 4)
    assert t.tolist() == [2.03, 4.0, 8.0] and sh[:, 0].tolist() == [1.0, 2.0, 3.0] and sc[1].tolist() == [0.0, 1.0]
    t, sc, sh, ps, pc = b.PresetTimeCallback([5.1], b.AffineAffect(1.0, 0.0, p_scale=2.0, p_shift=-0.5)).tables(2, 4)
    assert ps.shape == (1, 4) and (ps == 2.0).all() and (pc == -0.5).all() and (sc == 1.0).all()
    with pytest.raises(ValueError):
        b.PresetTimeCallback([1.0, 2.0], [b.AffineAffect(1.0, 0.0)]).tables(2, 4)
    prob = b.ODEProblem("lv", np.ones(2), (0.0, 10.0), np.array([1.5, 1.0, 3.0, 1.0]))
    ts = np.arange(0.0, 10.01, 0.5)
    with pytest.raises(NotImplementedError):          # a callback of another kind
        b.solve(b.EnsembleProblem(prob), b.Tsit5(adaptive=True), b.EnsembleB200(), trajectories=2, saveat=ts, callback=lambda integrator: None)
    with pytest.raises(NotImplementedError):          # extra saved points are not carried
        b.solve(b.EnsembleProblem(prob), b.Tsit5(adaptive=True), b.EnsembleB200(), trajectories=2, saveat=ts,
                callback=b.PresetTimeCallback([5.0], b.AffineAffect(1.0, 0.0), save_positions=(True, True)))
    with pytest.raises(NotImplementedError):          # a stepper without an event path
        b.solve(b.EnsembleProblem(prob), b.Rosenbrock23(), b.EnsembleB200(), trajectories=2, saveat=ts, abstol=1e-6, reltol=1e-6,
                callback=b.PresetTimeCallback([5.0], b.AffineAffect(1.0, 0.0)))


def _build_c_demo(tmp_path):
    import subprocess
    exe = str(tmp_path / "c_abi_demo")
    pkg = os.path.join(ROOT, "scimlsensitivity.jl_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "c_abi_demo.c"),
                           "-o", exe, "-L", pkg, "-lb200adj", "-Wl,-rpath," + pkg, "-lm"])
    return subprocess.run([exe], capture_output=True, text=True)


def test_header_is_plain_c_and_the_library_refuses_to_run_without_a_device(tmp_path):
    """include/b200adj.h compiles as C99 (-Wall -Wextra -Werror), a plain-C program links the library and drives the
    create / forward / reverse / destroy sequence of the Julia glue; on a machine without a GPU create answers
    B200ADJ_ERR_NO_DEVICE (exit code 3 of the demo) -- there is no CPU path to fall back to."""
    _lib.build()
    res = _build_c_demo(tmp_path)
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    assert res.returncode == (0 if has_gpu else 3), (res.returncode, res.stdout, res.stderr)
    if not has_gpu:
        assert "no CPU fallback" in res.stdout


@pytest.mark.gpu
def test_plain_c_program_computes_a_gradient_through_the_abi(tmp_path):
    """examples/c_abi_demo.c on the device: Lorenz N = 256, GaussAdjoint, host buffers; its printed dG/dp against the oracle."""
    from oracle import oracle as O
    res = _build_c_demo(tmp_path)
    assert res.returncode == 0, (res.stdout, res.stderr)
    line = [l for l in res.stdout.splitlines() if l.startswith("dG/dp")][0]
    dp = np.array([float(x) for x in line.split("(")[1].split(")")[0].split(",")])
    N = 256
    saveat = 0.1 * np.arange(11)
    u0 = np.stack([1.0 + 0.001 * np.arange(N), np.zeros(N), np.zeros(N)])
    cfg = O.make_cfg("lorenz", "gauss", "tsit5_fixed", N, saveat, 0.0, 1.0, dt=0.01, cost=("affine", 1.0, -2.0))
    ref = O.gradient(cfg, saveat, u0, np.array([10.0, 28.0, 8.0 / 3.0]))
    assert np.allclose(dp, ref["dp"], rtol=1e-9), (dp, ref["dp"])


def test_callback_family_host_objects():
    """The host objects of the callback families: the dosing affect's table follows the event-time order, the continuous callback's
    cache key tells the family extensions apart (a reused handle must not serve a different callback)."""
    cb = b.PresetTimeCallback([8.0, 3.0], [b.AffineAffect(1.0, 0.0, add_comp=0, add_param=1, add_coef=1.0), b.AffineAffect(0.5, 1.0)])
    comp, par, coef = cb.param_shift()
    assert comp.tolist() == [-1, 0] and par.tolist() == [0, 1] and coef.tolist() == [1.0, 1.0] and comp.dtype == np.int32
    assert b.PresetTimeCallback([1.0], b.AffineAffect(1.0, 0.0)).param_shift() is None
    base = b.ContinuousCallback(idx=0, direction=-1, p_comp=1, p_param=1, p_sign=-1.0)
    keys = {base.key(), b.ContinuousCallback(idx=0, direction=-1, p_comp=1, p_param=1, p_sign=-1.0, level_param=0, level_coef=0.75).key(),
            b.ContinuousCallback(idx=0, direction=-1, p_comp=1, p_param=1, p_sign=-1.0, add_comp=0, add_param=1, add_coef=1.0).key(),
            b.ContinuousCallback(idx=0, direction=-1, sq_comp=1).key(), b.ContinuousCallback(idx=0, direction=-1, sq_comp=1, sq_coef=2.0).key()}
    assert len(keys) == 5
    assert "relax" in b.FAMILIES if hasattr(b, "FAMILIES") else True


def test_bench_secondary_specs_are_consistent_with_the_oracle():
    """bench.py's secondary legs: every spec builds an oracle cfg (the parity checker) and its roofline closure returns a fraction."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    from oracle import oracle as O
    for mk in (bench.spec_c1, bench.spec_c3, bench.spec_c5):
        sp = mk()
        n = 4
        u0, p = sp["inputs"](n, 0)
        shared = sp.get("shared_p", True)
        cfg = O.make_cfg(sp["family"], sp["sensealg"], sp["stepper"], n, sp["saveat"], 0.0, sp["T"], dt=sp["dt"],
                         cost=("affine",) + tuple(sp["cost"]), shared_p=shared, **sp["okw"])
        dW = None
        if sp["stepper"] == "em":
            dW = np.sqrt(sp["dt"]) * np.random.default_rng(0).standard_normal((int(round(sp["T"] / sp["dt"])), 2, n))
        ref = O.gradient(cfg, sp["saveat"], u0, p, dW=dW, want_saved=False)
        assert np.isfinite(ref["dp"]).all() and ref["dp"].shape == ((sp["okw"].get("P", len(p)),) if shared else (p.shape[0], n))
        rf = sp["roofline"](n, 100.0, 1e-3, 6570.0, 1426.0)
        assert 0.0 < rf["frac"] < 10.0 and sp["cpu_sample"] >= sp["parity_members"]


def test_bench_dump_outputs_stays_within_64_mb(tmp_path):
    """bench.py --dump-outputs: dp whole, du0 whole while it fits, else every k-th member for the smallest k that fits; the
    flag is refused where there is no C2 device run to dump, and --steps below 1 is refused."""
    import importlib.util
    import subprocess
    import sys
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    dp = np.array([1.0, 2.0, 3.0])
    du0 = np.arange(3 * 3_000_000, dtype=np.float64).reshape(3, -1)            # 72 MB
    bench.dump_outputs(str(tmp_path), du0, dp)
    assert np.array_equal(np.load(tmp_path / "dp.npy"), dp)
    assert np.array_equal(np.load(tmp_path / "du0.npy"), du0[:, ::2])
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64e6
    bench.dump_outputs(str(tmp_path), du0[:, :1000], dp)
    assert np.array_equal(np.load(tmp_path / "du0.npy"), du0[:, :1000])
    for extra in (["--impl", "reference", "--dump-outputs", str(tmp_path)], ["--workload", "c1", "--dump-outputs", str(tmp_path)], ["--steps", "0"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert res.returncode == 2, (extra, res.stderr)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs first): exactly one JSON line on stdout with the contract's
    keys, measured on the oracle port; other ranks of a torchrun launch print nothing and exit 0."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--members", "128"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["metric"] == "ensemble adjoint trajectories/sec" and d["higher_is_better"] is True
    other = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--members", "128"],
                           capture_output=True, text=True, timeout=600, cwd=root, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert other.returncode == 0 and other.stdout.strip() == ""
