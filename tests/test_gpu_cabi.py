"""The C ABI driven from a plain-C program that samples on the GPU and is checked against the reference's own output
(tests/golden/unet64_default.npz).  Needs a B200, gcc and the CUDA runtime headers: `pytest -m gpu`."""
import os
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plain_c_program_samples_and_matches_reference(oracle, schedule, golden, tmp_path):
    from fastdiffsr_b200._lib import LIB_PATH
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if shutil.which("gcc") is None or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA runtime headers are missing")
    g = golden("unet64_default")
    sd = oracle.make_state_dict(oracle.DEFAULT_UNET, seed=0)        # the weights the fixture was generated with
    d = tmp_path
    with open(d / "manifest.txt", "w") as mf, open(d / "weights.bin", "wb") as wf:
        for k, v in sd.items():
            if k.startswith("denoise_fn."):
                a = np.ascontiguousarray(v.numpy(), dtype=np.float32)
                mf.write(f"{k} {a.size}\n")
                wf.write(a.tobytes())
    np.asarray(schedule["betas"], dtype=np.float64).tofile(d / "betas.bin")
    np.ascontiguousarray(g["cond"], dtype=np.float32).tofile(d / "cond.bin")
    np.ascontiguousarray(g["noises"], dtype=np.float32).tofile(d / "noise.bin")
    np.ascontiguousarray(g["sr"], dtype=np.float32).tofile(d / "sr_ref.bin")
    exe = str(d / "sample_check")
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(cuda, "include"), os.path.join(ROOT, "tests", "c_abi", "sample_check.c"),
                    "-o", exe, LIB_PATH, "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm",
                    "-Wl,-rpath," + os.path.dirname(LIB_PATH), "-Wl,-rpath," + os.path.join(cuda, "lib64")], check=True)
    res = subprocess.run([exe, str(d)], capture_output=True, text=True, timeout=300)
    print(res.stdout, res.stderr)
    assert res.returncode == 0, (res.returncode, res.stdout, res.stderr)
