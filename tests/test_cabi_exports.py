"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a,
loads, exports every symbol include/aligator_b200/gar.h declares, and its
no-compute helpers agree with the layout documented in the header."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    import aligator_b200.gar as gar
    return gar.lib()


def test_every_declared_symbol_is_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "aligator_b200", "gar.h")).read()
    names = sorted(set(re.findall(r"\b(ab2_gar_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n


def test_record_sizes_match_reference_layout(lib):
    """2nx^2 + 2nx*nu + nu^2 + 2nx + nu + nc(nx+nu+1) doubles (lqr-problem.hpp:60-65),
    padded to even; the BASELINE.md per-knot input counts."""
    import aligator_b200.gar as gar
    assert gar.stage_record_doubles(6, 3, 0) == 132
    assert gar.stage_record_doubles(12, 6, 0) == 498
    assert gar.stage_record_doubles(4, 2, 2) == 76
    assert gar.stage_record_doubles(14, 7, 0) == 672
    assert gar.stage_record_doubles(4, 2, 1) == 70  # 69 doubles, padded to even (16-byte TMA)
    assert gar.term_record_doubles(12, 0) == 156
    assert gar.term_record_doubles(4, 3) == 16 + 4 + 12 + 3


def test_supported_shapes(lib):
    import aligator_b200.gar as gar
    for shape in [(6, 3, 0, 6), (12, 6, 0, 12), (4, 2, 2, 4), (14, 7, 0, 14)]:
        assert gar.supported(*shape) == 1, shape   # compile-time shape, warp per instance
    assert gar.supported(57, 28, 0, 57) == 2      # BASELINE config 5: CTA per instance
    assert gar.supported(12, 6, 0, 30) == 2       # nx + nc0 exceeds the warp: CTA per instance
    assert gar.supported(7, 5, 3, 7) == 2         # arbitrary run-time shape
    assert gar.supported(120, 40, 0, 120) == 0    # does not fit one CTA's shared memory
    assert gar.supported(0, 1, 0, 0) == 0


def test_create_fails_loudly_without_cuda(lib):
    """No CPU fallback: without a CUDA device the handle cannot be created."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import aligator_b200.gar as gar
    with pytest.raises(gar.GarError):
        gar.CudaRiccatiBatch(12, 6, 0, 0, 12, 10, 4)


def test_unsupported_shape_is_an_error(lib):
    """Refused before any device is touched, so the same error with or without a GPU
    (57 x 28, BASELINE config 5, is a supported CTA-per-instance shape)."""
    import aligator_b200.gar as gar
    with pytest.raises(gar.GarError, match="does not fit one CTA"):
        gar.CudaRiccatiBatch(120, 40, 0, 0, 120, 10, 4)


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure; nothing under aligator_b200/ or include/ may
    reference it."""
    for base in ("aligator_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                    txt = open(os.path.join(dp, f)).read()
                    assert "gar_oracle" not in txt and "from oracle" not in txt, os.path.join(dp, f)
