"""The C++ drop-in boundary: seal/seal.h over libckks_b200.so.
CPU: the reference's own hot-path sources compile and link UNCHANGED against the shim.  GPU: a driver written
the way the reference writes its programs runs end to end through the shim.  The reference's sources are not
part of this repository: the tests that compile or run them read a checkout of MarwanNour/SEAL-FYP-Logistic-Regression
named by CKKS_REFERENCE_DIR (build() then also builds the reference programs into tests/cpp/_build/) and skip
without one."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "seal-fyp-logistic-regression_b200")
LIB = os.path.join(PKG_DIR, "libckks_b200.so")
INC = ["-I", os.path.join(ROOT, "include"), "-I", os.path.join(PKG_DIR, "include")]
REF = os.environ.get("CKKS_REFERENCE_DIR", "")
DRIVER = os.path.join(ROOT, "tests", "cpp", "shim_driver")

HOT_PATH_FILES = ["linear_transformation.cpp", "linear_transformation2.cpp", "polynomial.cpp",
                  "logistic_regression_ckks.cpp", "matrix_transpose.cpp", "matrix_multiplication.cpp",
                  "matrix_mult_benchmark.cpp", "4_ckks.cpp", "benchmark.cpp"]


def build_driver():
    src = os.path.join(ROOT, "tests", "cpp", "shim_driver.cpp")
    hdr = os.path.join(PKG_DIR, "include", "seal", "seal.h")
    if os.path.exists(DRIVER) and all(os.path.getmtime(DRIVER) >= os.path.getmtime(f) for f in (src, hdr, LIB)):
        return DRIVER
    subprocess.check_call(["g++", "-std=c++17", "-O2"] + INC + [src, "-o", DRIVER, LIB,
                                                              "-Wl,-rpath," + PKG_DIR])
    return DRIVER


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs CKKS_REFERENCE_DIR: a checkout of the reference's sources")
@pytest.mark.parametrize("name", HOT_PATH_FILES)
def test_reference_sources_build_unchanged(pkg, name, tmp_path):
    """`those files link against it unchanged` (BASELINE.json north_star): compile + link, no edits"""
    out = str(tmp_path / "a.out")
    res = subprocess.run(["g++", "-std=c++17", "-w", "-O0"] + INC + ["-I", REF, os.path.join(REF, name), "-o", out, LIB,
                                                                    "-Wl,-rpath," + PKG_DIR],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]


def test_shim_driver_builds(pkg):
    build_driver()
    assert os.path.exists(DRIVER)


@pytest.mark.gpu
def test_shim_driver_runs_on_gpu(pkg):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = build_driver()
    res = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and "OK" in res.stdout, res.stdout[-3000:]


REF_BUILD = os.path.join(ROOT, "tests", "cpp", "_build")


def _run_ref(name, cwd, stdin=None, timeout=600):
    exe = os.path.join(REF_BUILD, name)
    if not os.path.exists(exe):
        pytest.skip("reference binary %s was not prebuilt (build() builds it when CKKS_REFERENCE_DIR names the reference's sources)" % name)
    res = subprocess.run([exe], cwd=cwd, input=stdin, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    assert res.returncode == 0, res.stdout[-2000:]
    return res.stdout


@pytest.mark.gpu
def test_reference_matrix_mult_benchmark_runs_unmodified(pkg, tmp_path):
    """the reference's own matrix_mult_benchmark (CC_Matrix_Multiplication, d = 5, N = 16384), built
    unchanged against the shim, prints a decrypted product equal to its own plaintext check"""
    import re
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = _run_ref("matrix_mult_benchmark", str(tmp_path))
    got_blk = out.split("Resulting matrix:")[1].split("Expected Matrix:")[0]
    exp_blk = out.split("Expected Matrix:")[1]
    num = lambda t: [float(x) for x in re.findall(r"-?\d+\.\d+(?:e-?\d+)?", t)]
    got, exp = num(got_blk)[:25], num(exp_blk)[:25]
    assert len(got) == 25 and len(exp) == 25
    assert max(abs(a - b) for a, b in zip(got, exp)) < 1e-3


@pytest.mark.gpu
def test_reference_ckks_tutorial_runs_unmodified(pkg, tmp_path):
    """4_ckks.cpp (PI*x^3 + 0.4x + 1 with rescale / mod-switch / manual scale set)"""
    import re
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = _run_ref("4_ckks", str(tmp_path))
    exp = [float(x) for x in re.findall(r"-?\d+\.\d+", out.split("Expected result")[1].split("Computed result")[0])]
    got = [float(x) for x in re.findall(r"-?\d+\.\d+", out.split("Computed result")[1])][: len(exp)]
    assert len(exp) >= 6 and max(abs(a - b) for a, b in zip(got, exp)) < 1e-4


def test_batched_helper_header_compiles(pkg, tmp_path):
    """ckks_b200_helper.h (batched b200:: drop-ins for the reference's helper.h functions) is a
    self-contained header over seal/seal.h: it compiles and links without the reference tree"""
    src = tmp_path / "use_helper.cpp"
    src.write_text('#include "ckks_b200_helper.h"\n'
                   "int main() { auto f = &b200::Linear_Transform_Plain; auto g = &b200::cipher_dot_product;\n"
                   "auto h = &b200::C_Matrix_Encode; auto i = &b200::Linear_Transform_Cipher;\n"
                   "auto j = &b200::Linear_Transform_CipherMatrix_PlainVector; auto k = &b200::C_Matrix_Decode;\n"
                   "auto l = &b200::CC_Matrix_Multiplication; return (f && g && h && i && j && k && l) ? 0 : 1; }\n")
    res = subprocess.run(["g++", "-std=c++17", "-Wall", "-O0"] + INC + [str(src), "-o", str(tmp_path / "use_helper"), LIB,
                          "-Wl,-rpath," + os.path.dirname(LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]


@pytest.mark.gpu
def test_batched_helpers_bit_identical_to_reference_helpers(pkg, tmp_path):
    """tests/cpp/helper_driver.cpp: the reference's own Linear_Transform_Plain / _Cipher /
    _CipherMatrix_PlainVector / C_Matrix_Encode / cipher_dot_product (helper.h, compiled unchanged, one
    evaluator call at a time through the shim) against the batched b200:: versions on the same inputs and
    keys: every returned ciphertext is compared word for word"""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = _run_ref("helper_driver", str(tmp_path))
    assert "ALL BIT-IDENTICAL" in out and "MISMATCH" not in out, out[-2000:]
    assert out.count("bit-identical") == 6


@pytest.mark.gpu
def test_batched_matrix_multiplication_bit_identical_to_reference(pkg, tmp_path):
    """tests/cpp/matmul_driver.cpp: the reference's CC_Matrix_Multiplication (matrix_mult_benchmark.cpp,
    compiled unchanged with main() renamed) against b200::CC_Matrix_Multiplication, d = 4: same words"""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = _run_ref("matmul_driver", str(tmp_path))
    assert "ALL BIT-IDENTICAL" in out and "MISMATCH" not in out, out[-2000:]


def test_batched_lr_header_compiles(pkg, tmp_path):
    """ckks_b200_lr.h (b200::Horner_cipher / predict_cipher_weights / update_weights) compiles and links
    without the reference tree"""
    exe = str(tmp_path / "lr_driver")
    res = subprocess.run(["g++", "-std=c++17", "-Wall", "-O0"] + INC + [os.path.join(ROOT, "tests", "cpp", "lr_driver.cpp"), "-o", exe, LIB,
                          "-Wl,-rpath," + os.path.dirname(LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]


@pytest.mark.gpu
def test_cpp_lr_iteration_matches_plaintext(pkg, tmp_path):
    """tests/cpp/lr_driver.cpp: one encrypted training iteration through the C++ batched LR functions
    (b200::update_weights, 64 rows x 4 features, N = 32768, degree-3 Horner sigmoid): decrypted predictions and
    updated weights equal the plaintext computation within 1e-3"""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = os.path.join(REF_BUILD, "lr_driver")
    if not os.path.exists(exe):
        exe = str(tmp_path / "lr_driver")
        res = subprocess.run(["g++", "-std=c++17", "-O2"] + INC + [os.path.join(ROOT, "tests", "cpp", "lr_driver.cpp"), "-o", exe, LIB,
                              "-Wl,-rpath," + os.path.dirname(LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert res.returncode == 0, res.stdout[-3000:]
    res = subprocess.run([exe, "64"], cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and "LR OK" in res.stdout, res.stdout[-2000:]


def _build_host_checks(tmp_path):
    exe = str(tmp_path / "host_checks")
    res = subprocess.run(["g++", "-std=c++17", "-Wall", "-O0"] + INC + [os.path.join(ROOT, "tests", "cpp", "host_checks.cpp"), "-o", exe, LIB,
                          "-Wl,-rpath," + os.path.dirname(LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]
    return exe


def test_cpp_row_layout_matches_python(pkg, tmp_path):
    """b200::RowLayout / sigmoid_coeffs (ckks_b200_lr.h) pack exactly like lr.RowLayout / folded_coeffs"""
    import importlib
    import numpy as np
    lr = importlib.import_module("seal-fyp-logistic-regression_b200.lr")
    out = subprocess.run([_build_host_checks(tmp_path), "layout"], stdout=subprocess.PIPE, text=True, check=True).stdout
    rows = [np.array([float(x) for x in line.split()]) for line in out.strip().splitlines()]
    R, C = 5, 3
    X = np.array([[10 * i + j + 1 for j in range(C)] for i in range(R)], dtype=float)
    lay = lr.RowLayout(R, C, 16)
    assert np.array_equal(np.stack(rows[:R]), lay.rows(X))
    assert np.array_equal(np.stack(rows[R:R + C]), lay.columns(X))
    assert np.array_equal(rows[R + C], lay.weights(np.array([0.5, -1.5, 2.5])))
    assert np.array_equal(rows[R + C + 1], lay.labels(np.array([1, 0, 1, 1, 0.0])))
    for k, d in enumerate((3, 5, 7)):
        assert np.allclose(rows[R + C + 2 + k], lr.folded_coeffs(d), rtol=1e-15, atol=0)


def test_shim_fails_loudly_without_gpu(pkg, tmp_path):
    """no CPU fallback: on a machine without a CUDA device the first SEALContext::Create throws with the
    engine's message instead of computing anything on the host"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    res = subprocess.run([_build_host_checks(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 3 and "no CUDA device" in res.stdout, res.stdout


@pytest.mark.gpu
def test_cpp_column_layout_epoch_matches_plaintext(pkg, tmp_path):
    """tests/cpp/epoch_driver.cpp: the headline workload's op sequence (config 5: column layout, degree-7 tree
    sigmoid, per-feature cipher_dot_product chains in lock-step) driven from C++ through
    b200::column_epoch_gradient / apply_gradient, at a reduced size (64 samples, mini-batches of 16)"""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = os.path.join(REF_BUILD, "epoch_driver")
    if not os.path.exists(exe):
        exe = str(tmp_path / "epoch_driver")
        res = subprocess.run(["g++", "-std=c++17", "-O2"] + INC + [os.path.join(ROOT, "tests", "cpp", "epoch_driver.cpp"), "-o", exe, LIB,
                              "-Wl,-rpath," + os.path.dirname(LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert res.returncode == 0, res.stdout[-3000:]
    res = subprocess.run([exe, "64", "16", "1"], cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and "EPOCH OK" in res.stdout, res.stdout[-2000:]


# ---- SEAL binary serialization through the shim (SURVEY 8 row f2)
DUMP = os.path.join(ROOT, "tests", "cpp", "_build", "seal_dump_vectors")


def build_dump_tool():
    """tools/seal_dump_vectors.cpp is written against REAL SEAL 3.4.5 (it is the SEAL-side half of the cross-check); here it
    is compiled unchanged against the shim, which writes the same stream format"""
    src = os.path.join(ROOT, "tools", "seal_dump_vectors.cpp")
    hdr = os.path.join(PKG_DIR, "include", "seal", "seal.h")
    os.makedirs(os.path.dirname(DUMP), exist_ok=True)
    if os.path.exists(DUMP) and all(os.path.getmtime(DUMP) >= os.path.getmtime(f) for f in (src, hdr, LIB)):
        return DUMP
    subprocess.check_call(["g++", "-std=c++17", "-O2"] + INC + [src, "-o", DUMP, LIB, "-Wl,-rpath," + PKG_DIR,
                                                              "-Wl,-rpath,$ORIGIN/../../../seal-fyp-logistic-regression_b200"])
    return DUMP


def test_seal_dump_tool_builds_against_the_shim(pkg):
    build_dump_tool()
    assert os.path.exists(DUMP)


@pytest.mark.gpu
def test_seal_streams_written_by_the_shim_replay_bit_exact(pkg, po, tmp_path):
    """C++ (seal/seal.h shim: keygen, encrypt, evaluate, save) -> SEAL 3.4 binary files -> Python reader (sealio) -> the CUDA
    engine and the CPU oracle re-evaluate every op from the loaded inputs and keys -> identical to the saved outputs.
    With files from a real SEAL build in place of the shim's, the same command is the SEAL cross-check."""
    import sys
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = build_dump_tool()
    res = subprocess.run([exe, str(tmp_path), "12", "2"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:]
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "seal_replay.py"), str(tmp_path), "--backend", "both"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert res.returncode == 0 and "0 op(s) differ" in res.stdout, res.stdout[-3000:]
    assert res.stdout.count("bit-identical") == 20 and "hash convention confirmed" in res.stdout
