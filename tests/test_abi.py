"""The C-ABI library loads here (no GPU) and exports every symbol include/gibbs_b200.h declares."""
import ctypes as C
import os
import re

import pytest

from gibbssampling_b200 import _abi, _build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "gibbs_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gibbs_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_in_tree():
    assert os.path.exists(_build.LIB_PATH), "run __graft_entry__.build()"
    assert os.path.dirname(_build.LIB_PATH).endswith("gibbssampling_b200")


def test_every_source_file_is_a_build_dependency():
    """build() without force rebuilds only when a file in DEPS is newer than the library: an edit to a source missing
    from DEPS would leave the old library in place."""
    sources = {os.path.join(_build.CSRC, f) for f in os.listdir(_build.CSRC) if f.endswith((".cu", ".cuh", ".inc"))}
    assert sources - set(_build.DEPS) == set()


def test_every_declared_symbol_is_exported():
    lib = _abi.load()
    declared = _declared_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in gibbs_b200.h but not exported"
    assert sorted(_abi.EXPORTS) == declared


def test_struct_layouts_match_the_header():
    # gibbs_params: 2*int32 + 6 doubles + 4*int32; gibbs_run_stats: 5*int64 + 2*int32 + double
    assert C.sizeof(_abi.Params) == 8 + 6 * 8 + 24
    assert C.sizeof(_abi.RunStats) == 6 * 8 + 16 + 8
    assert _abi.Params.bg.offset == 16 and _abi.Params.cutoff.offset == 48 and _abi.Params.sampler.offset == 56


def test_abi_version_and_error_text():
    lib = _abi.load()
    assert lib.gibbs_abi_version() == 2
    assert isinstance(lib.gibbs_last_error(), bytes)


def test_no_cpu_fallback_without_a_device():
    """Without a CUDA device the product path must fail loudly (GIBBS_ERR_CUDA), never compute on the CPU."""
    lib = _abi.load()
    if lib.gibbs_device_count() > 0:
        pytest.skip("a CUDA device is present")
    from gibbssampling_b200.engine import GibbsEngine
    with pytest.raises(_abi.GibbsCudaError) as ei:
        GibbsEngine([b"ACGTACGT", b"ACGTACGT"])
    assert ei.value.code == _abi.GIBBS_ERR_CUDA
    assert "no CPU fallback" in str(ei.value)
    from gibbssampling_b200 import SiteSampler
    from gibbssampling_b200.CompositeVector import ProbabilityCompositeVector
    with pytest.raises(_abi.GibbsCudaError):
        SiteSampler.doSiteSamplingWithBPV(4, 1e-4, list("ATGC-"), ["ACGTACGT", "ACGTTTTT"],
                                          ProbabilityCompositeVector.ofACGT(.25, .25, .25, .25), seed=1)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gibbssampling_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle_lib" not in text and "gibbs_oracle" not in text, f


def test_constants_of_the_python_binding_match_the_header():
    """every #define GIBBS_* <integer> of include/gibbs_b200.h that _abi.py mirrors carries the same value (options, init
    paths, error codes, phases ...): a constant added on one side only is caught here, without a GPU"""
    text = open(os.path.join(ROOT, "include", "gibbs_b200.h")).read()
    defines = {m.group(1): int(m.group(2), 0) for m in re.finditer(r"^#define\s+(GIBBS_[A-Z0-9_]+)\s+(-?(?:0x[0-9a-fA-F]+|\d+))\s*(?:/\*.*)?$", text, flags=re.M)}
    assert {"GIBBS_OPT_INIT_PATH", "GIBBS_OPT_TILE_ROWS", "GIBBS_INIT_TILED", "GIBBS_INIT_SMEM"} <= set(defines)
    mirrored = [name for name in defines if hasattr(_abi, name)]
    assert len(mirrored) >= 18
    for name in mirrored:
        assert getattr(_abi, name) == defines[name], name
    for name in defines:
        if name.startswith(("GIBBS_OPT_", "GIBBS_INIT_")):
            assert hasattr(_abi, name), f"{name} is in the header but not in _abi.py"
