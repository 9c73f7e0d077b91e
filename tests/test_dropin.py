"""The C++ drop-in class (include/pqp_base_solver.hpp) driven like PathOptimizer::optimizePath.

CPU: it compiles against stub boundary types, links the C ABI library, and — with no GPU —
both calls return false with the library's error text (no CPU fallback).
GPU: its two-solve result equals the Python binding's on the same inputs, and the Cartesian
epilogue equals the oracle's restatement of getOptimizedPath."""
import math
import os
import subprocess

import numpy as np
import pytest

from path_optimizer_2_b200 import abi, solver, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "dropin_test")


BIN_REAL = BIN + "_real"
REF_STAGED = os.path.join(ROOT, "oracle", "_ref")


def _build(real=False):
    """real=True: bind the drop-in to the original project's OWN boundary types (data_struct.hpp,
    vehicle_state_frenet.{hpp,cpp} compile standalone, SURVEY.md §8c), staged in oracle/_ref/ by
    `make -C oracle ref` (build() does that where a checkout of that project is readable); None where
    nothing was staged."""
    solver.build_library()
    out = BIN_REAL if real else BIN
    src = os.path.join(ROOT, "tests", "cpp", "dropin_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "pqp_base_solver.hpp"), os.path.join(ROOT, "tests", "cpp", "ref_stub.hpp"),
            solver.LIB_PATH]
    if real:
        staged = [os.path.join(REF_STAGED, "include", "data_struct", h) for h in ("data_struct.hpp", "vehicle_state_frenet.hpp")]
        staged.append(os.path.join(REF_STAGED, "vehicle_state_frenet.o"))
        if not all(os.path.exists(f) for f in staged):
            return None
        deps += staged
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        extra = ["-DPQP_TEST_REAL_TYPES", "-I", os.path.join(REF_STAGED, "include"), "-w", staged[-1]] if real else ["-Wall"]
        subprocess.check_call(["g++", "-std=c++11", "-O1", "-o", out, src] + extra + [
            solver.LIB_PATH, "-Wl,-rpath," + os.path.dirname(solver.LIB_PATH)])
    return out


def _write_instance(path, knots, inst, n, ref, target_heading, constraint_end_heading=1):
    with open(path, "w") as f:
        f.write("%d\n" % n)
        for i in range(n):
            f.write(" ".join("%.17g" % v for v in (
                knots[abi.F_S, i], knots[abi.F_KREF, i], ref[0, i], ref[1, i], ref[2, i],
                knots[abi.F_B0_LB, i], knots[abi.F_B0_UB, i], knots[abi.F_B1_LB, i], knots[abi.F_B1_UB, i])) + "\n")
        f.write("%.17g %.17g %.17g %.17g\n%d\n" % (inst[abi.I_L0], inst[abi.I_PSI0], inst[abi.I_K0],
                                                   target_heading, constraint_end_heading))


@pytest.mark.parametrize("real", [False, True])
def test_dropin_compiles_and_fails_loudly_without_gpu(tmp_path, real):
    exe = _build(real)
    if exe is None:
        pytest.skip("the drop-in against the original project's types was not built (nothing staged in oracle/_ref)")
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    knots, inst, n, ref = synthetic.make_instance(3, 0, 60)
    p = str(tmp_path / "inst.txt")
    _write_instance(p, knots, inst, n, ref, 0.0)
    out = subprocess.run([exe, p], capture_output=True, text=True, check=True).stdout
    assert out.startswith("solve 0 ") and "no CUDA device" in out


@pytest.mark.gpu
@pytest.mark.parametrize("real", [False, True])
def test_dropin_matches_python_binding(tmp_path, real):
    from oracle import oracle
    exe = _build(real)
    if exe is None:
        pytest.skip("the drop-in against the original project's types was not built (nothing staged in oracle/_ref)")
    params = abi.default_params()
    for idx in range(3):
        knots, inst, n, ref = synthetic.make_instance(3, idx, 120)
        # target heading such that the signed <70deg test selects a +-0.087 box (base_solver.cpp:254-259)
        target_heading = ref[2, n - 1] + 0.05
        inst = inst.copy()
        e = (target_heading - ref[2, n - 1] + math.pi) % (2 * math.pi) - math.pi
        inst[abi.I_EPSI_LO], inst[abi.I_EPSI_HI] = e - 0.087, e + 0.087
        p = str(tmp_path / ("inst%d.txt" % idx))
        _write_instance(p, knots, inst, n, ref, target_heading)
        lines = subprocess.run([exe, p], capture_output=True, text=True, check=True).stdout.strip().split("\n")
        assert lines[0].startswith("solve 1 status 0"), lines[0]
        assert lines[1].startswith("resolve 1 status 0"), lines[1]
        got = np.array([[float(v) for v in ln.split()] for ln in lines[2:]])
        assert got.shape == (n, 7)
        hb = abi.HostBatch(knots[None], inst[None], np.array([n], dtype=np.int32))
        sv = solver.PathQpSolver(params, n_max=n, batch_max=1)
        r1 = sv.solve(hb)
        r2 = sv.resolve(hb.with_linearisation(r1.sol))
        sv.close()
        # identical inputs through the same library: bit-identical Frenet solution
        assert np.array_equal(got[:, 5], r2.sol[0, 0, :n]) and np.array_equal(got[:, 6], r2.sol[0, 1, :n])
        assert np.array_equal(got[:, 3], r2.sol[0, 2, :n]) and np.array_equal(got[:-1, 4], r2.sol[0, 3, :n - 1])
        xyh = oracle.frenet_to_cartesian(ref[:, :n], r2.sol[0, 0, :n], r2.sol[0, 1, :n])
        assert np.allclose(got[:, 0:3].T, xyh, atol=1e-12, rtol=0)


@pytest.mark.gpu
def test_dropin_long_path_and_handle_pool(tmp_path):
    """A 100 m plan (n = 400 > 255 knots: the reference sizes everything from input_path.size(),
    base_solver.cpp:15-39) through the drop-in, constructed per plan like the reference's caller
    (path_optimizer.cpp:138): the handle pool creates one handle and re-uses it for every later plan."""
    exe = _build(False)
    params = abi.default_params()
    knots, inst, n, ref = synthetic.make_instance(3, 1, 400)
    assert n == 400 and knots[abi.F_S, n - 1] > 60.0
    inst = inst.copy()
    inst[abi.I_EPSI_LO], inst[abi.I_EPSI_HI] = -abi.INFTY, abi.INFTY  # constraint_end_heading = 0 below
    p = str(tmp_path / "long.txt")
    _write_instance(p, knots, inst, n, ref, 0.0, constraint_end_heading=0)
    lines = subprocess.run([exe, p, "20"], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    assert lines[0].startswith("plans 21 "), lines[0]
    tok = lines[0].split()
    stats = {tok[i]: float(tok[i + 1]) for i in range(0, 10, 2)}
    assert stats["creates"] == 1 and stats["hits"] >= 20
    assert stats["later_ms"] < stats["first_ms"]
    assert lines[1].startswith("solve 1 status 0"), lines[1]
    assert lines[2].startswith("resolve 1 status 0"), lines[2]
    got = np.array([[float(v) for v in ln.split()] for ln in lines[3:]])
    hb = abi.HostBatch(knots[None], inst[None], np.array([n], dtype=np.int32))
    sv = solver.PathQpSolver(params, n_max=n, batch_max=1)
    r1 = sv.solve(hb)
    r2 = sv.resolve(hb.with_linearisation(r1.sol))
    sv.close()
    assert np.array_equal(got[:, 5], r2.sol[0, 0, :n]) and np.array_equal(got[:, 3], r2.sol[0, 2, :n])
    print("drop-in plan loop:", lines[0])
