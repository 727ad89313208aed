"""The per-substep loop of the highway step kernel has to stay near the 32 KB L1.5 instruction cache: cutting it from
70 KB to 32 KB was worth +9 % on the headline config (profiles/r2_kernel_history.md), and a stray inlined helper or
unrolled loop silently undoes that.  Cross-compiles hwy_highway.cu (no GPU needed) and measures the loop statically
with tools/loop_size.sh."""
import ast
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("nvcc") is None or shutil.which("nvdisasm") is None, reason="needs nvcc + nvdisasm")
def test_highway_substep_loop_fits_the_instruction_cache_budget(tmp_path):
    out = subprocess.run(["bash", os.path.join(ROOT, "tools", "loop_size.sh")], cwd=ROOT, capture_output=True, text=True,
                         timeout=600, env=dict(os.environ, HWY_LOOP_SIZE_DIR=str(tmp_path)))
    assert out.returncode == 0, out.stderr[-800:]
    line = [l for l in out.stdout.splitlines() if "backward spans:" in l][-1]
    total = int(line.split(" total ")[1].split(" B;")[0])
    spans = ast.literal_eval(line.split("backward spans:")[1].strip())
    # the big spans are the epilogue's (autoreset) jumps back across the whole function; the substep loop is the
    # largest one below 64 KB
    loop = max(s for s, _, _ in spans if s < 64 * 1024)
    assert 16 * 1024 < loop <= 36 * 1024, f"substep loop of highway_step_kernel<64, true> is {loop} B"
    assert total <= 170 * 1024, f"highway_step_kernel<64, true> is {total} B"
