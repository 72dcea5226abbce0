"""tests/test_zz_eco_gpu.py -- the `-m gpu` tests of the ECO entry points, most of which the round's GPU budget did not reach -- executed
here WITHOUT a GPU: a pytest subprocess with tests/cpu_emul/gpu_file_on_cpu_plugin.py, in which `pytracking_b200._lib.lib()` hands out
tests/cpu_emul/eco_abi_emul.cpp (the launchers csrc/eco_cg.cu and csrc/eco_loc.cu compiled verbatim as host code, the kernels run by the
SIMT shim with the 148-CTA launch of a B200) in place of libb200trk.so.  The same test code, `ops` wrappers, ctypes signatures, plug-in
seams, launch plans and kernels as on the device; what differs is who executes the kernels.  The two tracker-level tests (the unmodified
reference ECO tracker over 12 frames, stock vs above the engine; the plugin builds it on the CPU) take three more minutes and run only
with B200_ECO_TRACKER_ON_CPU=1, as do the two slowest full-size cases of the online kernel (the 63x32x200x16 block with streamed slabs:
a minute of emulation); the recorded run of all 43 is profiles/r02zc_eco_gpu_test_file_on_cpu.txt."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FULL = os.environ.get("B200_ECO_TRACKER_ON_CPU") == "1"


def test_eco_gpu_test_file_runs_on_the_cpu_against_launchers_and_kernel_sources(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    lib = str(tmp_path / "libeco_abi_emul.so")
    # -fsanitize=alignment (recovering: a report on stderr): every float2 / float4 access of the kernels aligned as the device requires,
    # for the shared-memory carving and the workspace layout of exactly the launches the GPU tests make
    cmd = ["g++", "-std=c++17", "-O2", "-g", "-pthread", "-shared", "-fPIC", "-fno-gnu-unique", "-ffp-contract=off", "-Wno-unknown-pragmas",
           "-DB200_EMUL_COOP_FIBERS", "-fsanitize=alignment", "-x", "c++", os.path.join(ROOT, "tests", "cpu_emul", "eco_abi_emul.cpp"), "-o", lib]
    if subprocess.run(cmd, capture_output=True).returncode != 0:
        cmd.remove("-fsanitize=alignment")
        subprocess.run(cmd, check=True, capture_output=True)
    env = dict(os.environ, B200_ECO_ABI_EMUL=lib, B200_EMUL_SMS="148",
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "tests", "cpu_emul"), ROOT, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_zz_eco_gpu.py"), "-p", "gpu_file_on_cpu_plugin", "-q", "-x",
                        "-rs", "-p", "no:cacheprovider", "-s"] + ([] if FULL else ["-k", "not tracker and not 63-32-200-16-200 and not 17-9-200-32-37"]), capture_output=True, text=True, env=env, cwd=ROOT, timeout=3000)
    tail = r.stdout[-3000:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert "runtime error" not in r.stderr and "runtime error" not in r.stdout, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail
    n = int(r.stdout.strip().split("\n")[-1].split(" passed")[0].split()[-1])
    # the tests that run the reference pytracking package itself skip where no pytracking checkout is importable; nothing else may skip
    skips = [l for l in r.stdout.splitlines() if l.startswith("SKIPPED")]
    assert all("reference tree not staged" in l for l in skips), tail
    n_no_reference = sum(int(l.split("[", 1)[1].split("]", 1)[0]) for l in skips)
    assert n + n_no_reference >= (43 if FULL else 39), tail                                            # 13 golden runs of the online kernel + everything that had not run on a B200
