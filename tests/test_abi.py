"""CPU: the C-ABI library loads, exports every symbol include/b2pn.h declares, and the grouping
kernels' SASS keeps the bit-exact arithmetic contract (no fused multiply-add)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b2pn.h")


@pytest.fixture(scope="module")
def built_lib():
    from dl_biomass_b200 import _lib
    _lib.build()
    return _lib


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2pn_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound(built_lib):
    names = declared_symbols()
    assert "b2pn_fps_f32" in names and "b2pn_ball_query_f32" in names
    nm = subprocess.run(["nm", "-D", "--defined-only", built_lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (b2pn_[a-z0-9_]+)", nm))
    assert set(names) <= exported, sorted(set(names) - exported)
    assert set(names) == set(built_lib.SIGNATURES), "ctypes table and header disagree"
    h = built_lib.lib()
    assert h.b2pn_abi_version() == built_lib.ABI_VERSION
    assert h.b2pn_fps_num_samples(7168, 0.2) == 1434
    assert b"invalid" in h.b2pn_error_string(-1)


def test_argument_errors_need_no_gpu(built_lib):
    h = built_lib.lib()
    assert h.b2pn_fps_f32(None, None, None, None, 2, 10, None, None, None, None, None) == -1
    assert h.b2pn_fps_f32(None, None, None, None, 0, 0, None, None, None, None, None) == 0
    import ctypes
    bad = built_lib.FpsOptions(3, 0, 0, None)                 # no such cluster size
    assert h.b2pn_fps_f32(None, None, None, None, 0, 0, None, None, None, ctypes.byref(bad), None) == -1
    assert 0 <= h.b2pn_fps_random_start(7, 0, 3, 1000) < 1000 and h.b2pn_fps_random_start(7, 0, 3, 0) == -1
    assert h.b2pn_adam_step(None, None, None, None, 8, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None, None) == -1
    assert h.b2pn_adam_step(None, None, None, None, 6, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None, None) == -1   # n % 4
    assert h.b2pn_adam_step(None, None, None, None, 0, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, None, None) == 0
    assert h.b2pn_ball_query_f32(None, None, None, None, 1, 5, 5, 2.0, 64, None, None, None) == -1
    assert h.b2pn_ball_query_f32(None, None, None, None, 1, 5, 5, 2.0, 0, None, None, None) == -1


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "dl_biomass_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "libb2pn_oracle" not in txt, f


def test_oracle_never_imports_product():
    """The oracle is an independent restatement: oracle/ref.py and oracle/augment_ref.py must not lean on the package they
    check (the golden-vector generator scripts may use its synthetic-cloud helper)."""
    for f in ("ref.py", "augment_ref.py", "b2pn_oracle.c"):
        txt = open(os.path.join(ROOT, "oracle", f)).read()
        assert not re.search(r"^\s*(from|import)\s+dl_biomass_b200\b", txt, flags=re.M), f
        assert "libb2pn.so" not in txt, f


def test_cpu_tensors_fail_loudly(built_lib):
    import torch
    from dl_biomass_b200 import ops
    lv = ops.build_levels([10], [0.5], torch.device("cpu"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.fps(torch.zeros(10, 3), lv[0], lv[1])


def test_grouping_sass_has_no_fma(built_lib):
    """Distances must be ((dx*dx+dy*dy)+dz*dz) with separate roundings (SURVEY.md A.7)."""
    sass = subprocess.run([built_lib.cuda_tool("cuobjdump"), "-sass", built_lib.LIB_PATH], capture_output=True,
                          text=True).stdout
    cur, bad = None, []
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
        elif cur and ("fps_kernel" in cur or "ball_query_kernel" in cur) and re.search(r"\bFFMA2?\b", line):
            # (the Morton-sorted FPS variants and the grid ball query compute their distances with the same
            #  __f*_rn intrinsics; their cell / Morton quantisation legitimately uses FMA and is not checked here)
            bad.append((cur, line.strip()))
        elif cur and "fps_f64_kernel" in cur and re.search(r"\bDFMA\b", line):
            bad.append((cur, line.strip()))
    assert not bad, bad[:3]
    assert "FMUL2" in sass and "FADD2" in sass and "REDUX" in sass


def test_host_side_sizing_helpers(built_lib):
    """Host-only entry points: capacity / workspace bounds and argument checks (no GPU involved)."""
    import ctypes
    h = built_lib.lib()
    # compacted-row capacity: never below the slots in use, grows with n_dst, rejects K > 64
    for n_dst, K in ((1, 64), (24000, 64), (6000, 64), (1000, 16), (1000, 40), (7, 8)):
        cap = h.b2pn_pack_rows_capacity(n_dst, K)
        assert cap % 128 == 0 and cap >= n_dst * min(64, (K + 7) // 8 * 8) // max(1, 64 // ((K + 7) // 8 * 8)) // 64 * 64
        assert h.b2pn_pack_rows_capacity(n_dst + 64, K) >= cap
    assert h.b2pn_pack_rows_capacity(10, 128) == -2          # B2PN_ENOTSUP
    assert h.b2pn_pack_rows_capacity(-1, 64) == -1           # B2PN_EINVAL
    assert h.b2pn_pack_rows_workspace_bytes(24000) >= 24000 * 4
    assert h.b2pn_ball_query_workspace_bytes(12, 120000) >= 120000 * 4 + 12 * 8192 * 4
    assert h.b2pn_ball_query_workspace_bytes(-1, 10) == -1
    neg = built_lib.SaArgs()                                  # launch options are per-call fields, checked per call
    neg.precision, neg.sm_limit = 1, -3
    assert h.b2pn_sa_forward(ctypes.byref(neg), None) == -1 and h.b2pn_sa_workspace_bytes(ctypes.byref(neg), 0) == -1
    nm = subprocess.run(["nm", "-D", "--defined-only", built_lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "b2pn_set_" not in nm and "set_variant" not in nm   # no process-wide setters left in the ABI
    assert h.b2pn_head_forward(None, None) == -1 and h.b2pn_head_backward(None, None, None) == -1
    assert h.b2pn_sa_gather_rows(None, None) == -1
    sa_args = built_lib.SaArgs()                              # fp32 levels gather inside their loaders
    assert h.b2pn_sa_gather_rows(ctypes.byref(sa_args), None) == -2
    a = built_lib.HeadArgs()
    a.B = 40                                                  # more rows than the fused head takes
    for i, c in enumerate((1024, 128, 128, 4)):
        a.c[i] = c
    assert h.b2pn_head_forward(ctypes.byref(a), None) == -2
