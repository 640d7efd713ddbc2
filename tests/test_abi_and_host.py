"""CPU-side checks: the C-ABI library loads and exports every symbol include/cpcsv.h declares
(no compute calls), argument errors are reported without a GPU, and the product refuses to
run on CPU tensors (no fallback)."""
import os
import re

import pytest
import torch

from cpcsv_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    header = open(os.path.join(ROOT, "include", "cpcsv.h")).read()
    declared = set(re.findall(r"\b(cpcsv_[a-z0-9_]+)\s*\(", header))
    declared -= {"cpcsv_stream_t"}
    lib = _lib.load()
    bound = set(_lib.SIGNATURES) | set(_lib.OTHER_SYMBOLS)
    assert declared == bound, (declared - bound, bound - declared)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.cpcsv_version() >= 100


def test_argument_errors_do_not_need_a_gpu():
    lib = _lib.load()
    rc = lib.cpcsv_bn_stats(None, 0, 0, 0, None, None)
    assert rc < 0 and b"bn_stats" in lib.cpcsv_last_error_string()
    g = _lib.Gemm()
    g.mode = 7
    assert lib.cpcsv_conv_gemm(g, None) < 0
    assert b"mode" in lib.cpcsv_last_error_string()


def test_no_cpu_fallback():
    x = torch.zeros(8, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.bn_stats(x, torch.zeros(16, dtype=torch.float64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.tanh_fwd(x, x)


def test_gemm_struct_layout_matches_header():
    # sizeof(cpcsv_gemm_t): 19 int32, 4 int64, 3 pointers + stats_ld, 4 views (88 B), 16 taps (40 B)
    import ctypes as C
    assert C.sizeof(_lib.View5) == 8 + 5 * 8 + 5 * 8
    assert C.sizeof(_lib.Tap) == 40
    # 19 int32 fields (incl. cta_pair) padded to 20 x 4 bytes before the int64 members
    assert C.sizeof(_lib.Gemm) == 20 * 4 + 4 * 8 + 2 * 8 + 2 * 8 + 4 * 88 + 16 * 40
    assert C.sizeof(_lib.AdamHyper) == 2 * 8 + 3 * 8 and C.sizeof(_lib.AdamTensor) == 40 and C.sizeof(_lib.Plane) == 32


def test_miscc_package_falls_through_to_the_reference_for_modules_it_does_not_replace(tmp_path):
    """with this package first on sys.path, ``from miscc.datasets import ...`` (reference
    main_pororo.py:23, inference.py:26) still finds the reference's own miscc/datasets.py"""
    import subprocess
    import sys
    ref = tmp_path / "ref" / "miscc"
    ref.mkdir(parents=True)
    (ref / "__init__.py").write_text("")
    (ref / "datasets.py").write_text("class TextDataset:\n    origin = 'reference'\n")
    (ref / "utils.py").write_text("raise RuntimeError('the reference utils must stay shadowed')\n")
    pkg = os.path.join(ROOT, "cpcstoryvisualization-pytorch_b200")
    code = ("import sys; sys.path[:0] = [%r, %r]; from miscc.datasets import TextDataset; import miscc.utils as u; "
            "print(TextDataset.origin, hasattr(u, 'compute_discriminator_loss'))" % (pkg, str(tmp_path / "ref")))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.split()[-2:] == ["reference", "True"]


def test_weight_cache_entries_die_with_their_parameter():
    """keys carry id(param): a recycled id / address / version of a freed parameter must not hit the
    old entry, and the packed planes must not outlive the parameter"""
    import gc
    from cpcsv_b200 import engine
    cache = engine.WeightCache()
    built = []

    def get(p):
        return cache.get((id(p), "k"), p, lambda: built.append(1) or torch.zeros(3))
    a = torch.nn.Parameter(torch.zeros(4))
    get(a)
    get(a)
    assert len(built) == 1 and len(cache.d) == 1
    key = next(iter(cache.d))
    del a
    gc.collect()
    assert len(cache.d) == 0
    # an impostor with the same key and tag (what id / address recycling would produce) is rebuilt
    b = torch.nn.Parameter(torch.zeros(4))
    get(b)
    ent = cache.d[(id(b), "k")]
    c = torch.nn.Parameter(torch.zeros(4))
    import weakref
    cache.d[(id(b), "k")] = engine.CacheEntry(ent.tag, ent.val, ent.stream, ent.event, weakref.ref(c))
    n = len(built)
    get(b)
    assert len(built) == n + 1
    del key


def test_first_discriminator_layer_past_its_kernel_limit_is_refused(monkeypatch):
    """layer 0 of a discriminator is one direct kernel (csrc/enc0.cu) for at most 128 output channels:
    DF_DIM 160 (padded to 192) raises instead of running some other path"""
    import emulator
    import harness
    from oracle import params, presets
    emulator.install(monkeypatch)
    p = presets.get("tiny", DF_DIM=160)
    D = harness.build_product(p, params.init_all(p, 0), torch.device("cpu"))["D_im"]
    with pytest.raises(NotImplementedError, match="at most 128 output channels"):
        D(torch.zeros(p["IM_BATCH"], 3, 64, 64))
