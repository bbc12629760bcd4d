"""CPU: the drop-in matmul.h keeps the reference's struct layout (field order / offsets) so reference call sites
link against it unchanged.  Checked by compiling a probe against this header and comparing its sizes and offsets with what
the same probe printed for the reference's kernels/matmul.h (-DQM_CUDA), recorded in tests/golden/matmul_h_layout.txt by make_golden.py."""
import subprocess
import tempfile
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
PROBE = r'''
#include <cstdio>
#include <cstddef>
#include MATMUL_H
int main() {
    printf("%zu %zu %zu %zu ", sizeof(matrix), sizeof(matmul_params), sizeof(quantization_params), sizeof(optimization_params));
    printf("%zu %zu %zu %zu %zu ", offsetof(matrix, half_data_ptr), offsetof(matrix, int32_data_ptr), offsetof(matrix, int8_data_ptr), offsetof(matrix, int4_data_ptr), offsetof(matrix, qparams));
    printf("%zu %zu %zu %zu %zu %zu %zu\n", offsetof(matmul_params, bias), offsetof(matmul_params, alpha), offsetof(matmul_params, half_alpha), offsetof(matmul_params, half_scales),
           offsetof(matmul_params, int32_zero_point), offsetof(matmul_params, block_size), offsetof(matmul_params, A_scales));
    return 0;
}
'''


def probe(header: str, extra):
    with tempfile.TemporaryDirectory() as d:
        src = Path(d) / "p.cu"
        src.write_text(PROBE.replace("MATMUL_H", f'"{header}"'))
        exe = Path(d) / "p"
        subprocess.run(["nvcc", "-std=c++17", "-w", "-o", str(exe), str(src)] + extra, check=True, capture_output=True)
        return subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip()


def test_struct_layout_matches_reference(golden_dir):
    ours = probe(str(ROOT / "tinychatengine_b200/host/matmul.h"), [])
    ref = (golden_dir / "matmul_h_layout.txt").read_text().strip()
    assert ours == ref, (ours, ref)
    assert len(ours.split()) == 16
