"""Host emulation of the diagonal-tile program of the blocked Cholesky (csrc/ba_tile.cuh): the template the CUDA
kernel instantiates is run on the CPU with the 512 threads of each CTA executed phase by phase in forward, reversed
and shuffled order (tests/tile_emulation.cc). Checks the factor and the inverse against plain loops, that the result
does not depend on the thread order inside a phase (barrier placement), the identity padding of partial tiles and
the indefinite-pivot flag. No GPU involved."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_tile_program_on_the_host(tmp_path):
    exe = str(tmp_path / "b200ba_tile_emulation")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wno-unknown-pragmas",
                           os.path.join(ROOT, "tests", "tile_emulation.cc"), "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "TILE_EMULATION_OK" in r.stdout
