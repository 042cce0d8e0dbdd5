"""CPU-side checks of the drop-in boundary: the library builds/loads, exports every symbol that
include/vlg_b200.h declares, the ctypes mirror of vlg_problem_t matches the C layout, and argument
validation works without a GPU (no compute call is made here)."""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vlg_b200.h")

import vlg_b200  # noqa: E402
from vlg_b200 import _cabi  # noqa: E402


def _declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vlg_[a-z_0-9]+)\s*\(", text)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _cabi.load()
    declared = _declared_symbols()
    assert set(declared) == set(_cabi.EXPORTS), (declared, _cabi.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.vlg_version() == 200 == _cabi.ABI_VERSION


FIELDS = ["struct_size", "abi_version", "N", "H", "W", "K", "dtype", "padding", "coord_mode", "flags", "ignore_index", "w_l1", "w_gd",
          "w_ssim", "w_ce", "w_tv", "term_mask", "ce_norm", "global_N", "ce_class_weight"]


def _c_layout():
    """sizeof(vlg_problem_t) and the offset of every field, from the header as gcc compiles it."""
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "vlg_b200.h"
int main(void){
  printf("%zu", sizeof(vlg_problem_t));
#define O(f) printf(" %zu", offsetof(vlg_problem_t, f));
  FIELDS
  return 0; }
'''.replace("FIELDS", " ".join(f"O({f})" for f in FIELDS))
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        return [int(v) for v in subprocess.check_output([exe]).split()]


def test_problem_struct_layout_matches_c():
    vals = _c_layout()
    P = _cabi.Problem
    assert [n for n, _ in P._fields_] == FIELDS
    assert vals[0] == C.sizeof(P)
    assert vals[1:] == [getattr(P, n).offset for n in FIELDS]
    assert P().struct_size == vals[0] and P().abi_version == _cabi.ABI_VERSION


def test_python_constants_match_the_header():
    """Every VLG_FLAG_* / VLG_TERM_* / VLG_STATUS_* / VLG_CE_NORM_* / VLG_NEAR_RADIUS the Python side mirrors has the
    value the header (as gcc sees it) gives it -- a flag added on one side only would silently select another path."""
    names = {"VLG_FLAG_NO_FAR_PATH": _cabi.FLAG_NO_FAR_PATH, "VLG_FLAG_NO_TMA": _cabi.FLAG_NO_TMA,
             "VLG_FLAG_PASS2_COORDS": _cabi.FLAG_PASS2_COORDS, "VLG_FLAG_FAR_WIDE": _cabi.FLAG_FAR_WIDE,
             "VLG_TERM_L1": _cabi.TERM_L1, "VLG_TERM_GD": _cabi.TERM_GD, "VLG_TERM_SSIM": _cabi.TERM_SSIM,
             "VLG_TERM_CE": _cabi.TERM_CE, "VLG_TERM_TV": _cabi.TERM_TV,
             "VLG_STATUS_BAD_LABEL": _cabi.STATUS_BAD_LABEL, "VLG_STATUS_FAR_TAPS": _cabi.STATUS_FAR_TAPS,
             "VLG_CE_NORM_TORCH": _cabi.CE_NORM_TORCH, "VLG_CE_NORM_COUNT": _cabi.CE_NORM_COUNT,
             "VLG_NEAR_RADIUS": _cabi.NEAR_RADIUS}
    src = '#include <stdio.h>\n#include "vlg_b200.h"\nint main(void){\n' + "".join(
        f'printf("%lld ", (long long)({n}));\n' for n in names) + "return 0; }\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, c])
        vals = [int(v) for v in subprocess.check_output([exe]).split()]
    assert dict(zip(names, vals)) == names
    flags = [v for n, v in names.items() if n.startswith("VLG_FLAG_")]
    assert len(set(flags)) == len(flags) and all(v & (v - 1) == 0 for v in flags), "flags are distinct single bits"


def test_integration_doc_binding_matches_c():
    """INTEGRATION.md shows a maintainer the ctypes mirror of vlg_problem_t: the DOCUMENT is what gets copied, so
    the snippet itself is executed here and its layout compared with the header (round 1 shipped a stale one)."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"class Problem\(C\.Structure\):.*?\n(?=\S)", text, flags=re.S)
    assert m, "INTEGRATION.md no longer contains the Problem mirror"
    ns = {"C": C}
    exec(m.group(0), ns)
    D = ns["Problem"]
    vals = _c_layout()
    assert [n for n, _ in D._fields_] == FIELDS
    assert C.sizeof(D) == vals[0]
    assert [getattr(D, n).offset for n in FIELDS] == vals[1:]


def test_stale_descriptor_is_refused():
    """A caller compiled against an older, shorter vlg_problem_t (or one that never set struct_size) is told so
    instead of having the library read past its buffer."""
    lib = _cabi.load()
    ok = _cabi.Problem(N=2, H=16, W=16, K=20, padding=1)
    assert lib.vlg_workspace_bytes(C.byref(ok), 0) > 0
    stale = _cabi.Problem(N=2, H=16, W=16, K=20, padding=1, struct_size=96)
    assert lib.vlg_workspace_bytes(C.byref(stale), 0) == 0
    assert b"struct_size" in lib.vlg_last_error()
    old = _cabi.Problem(N=2, H=16, W=16, K=20, padding=1, abi_version=100)
    assert lib.vlg_workspace_bytes(C.byref(old), 0) == 0
    assert b"abi_version" in lib.vlg_last_error()


def test_header_constants_match_binding():
    text = open(HEADER).read()
    consts = dict(re.findall(r"#define\s+(VLG_[A-Z0-9_]+)\s+\(?(-?\d+)u?\)?", text))
    assert int(consts["VLG_F32"]) == _cabi.F32 and int(consts["VLG_BF16"]) == _cabi.BF16
    assert int(consts["VLG_PAD_BORDER"]) == _cabi.PAD_BORDER
    assert int(consts["VLG_COORD_GRID"]) == _cabi.COORD_GRID
    assert int(consts["VLG_NEAR_RADIUS"]) == _cabi.NEAR_RADIUS
    assert int(consts["VLG_LOSS_SLOTS"]) == _cabi.LOSS_SLOTS
    assert int(consts["VLG_LOSS_TOTAL"]) == _cabi.LOSS_TOTAL
    assert int(consts["VLG_TERM_ALL"]) == _cabi.TERM_ALL


def test_argument_validation_without_gpu():
    lib = _cabi.load()
    bad = _cabi.Problem(N=1, H=1, W=8, K=20)
    assert lib.vlg_workspace_bytes(C.byref(bad), 0) == 0
    assert b"H>=2" in lib.vlg_last_error()
    badk = _cabi.Problem(N=1, H=8, W=8, K=7)
    assert lib.vlg_workspace_bytes(C.byref(badk), 0) == 0
    assert b"K=7" in lib.vlg_last_error()
    ok = _cabi.Problem(N=2, H=128, W=256, K=20, padding=1)
    small = lib.vlg_workspace_bytes(C.byref(ok), 0)
    big = lib.vlg_workspace_bytes(C.byref(ok), 1)
    P = 2 * 128 * 256
    assert 0 < small < big
    assert big >= P * 23 * 4 + P * 23 * 8
    ok.flags = _cabi.FLAG_NO_FAR_PATH
    assert lib.vlg_workspace_bytes(C.byref(ok), 1) < big
    # bits 4 and 8 selected pass-1 organisations that are retired; unknown bits are refused, not ignored
    for retired in (4, 8, 4 | 8, 128):
        unknown = _cabi.Problem(N=2, H=128, W=256, K=20, padding=1, flags=_cabi.FLAG_NO_TMA | retired)
        assert lib.vlg_workspace_bytes(C.byref(unknown), 0) == 0
        assert b"unknown flag bits" in lib.vlg_last_error()
        assert b"VLG_FLAG_TILE_RGB" in lib.vlg_last_error() and b"VLG_FLAG_TILE_LAYOUT" in lib.vlg_last_error()
    # NULL workspace is refused before anything is launched
    rc = lib.vlg_reduce_partials(C.byref(ok), None, None, 0, None)
    assert rc == -1


def test_no_cpu_fallback():
    import torch
    x = torch.zeros(1, 3, 8, 8)
    with pytest.raises(vlg_b200.VlgError):
        vlg_b200.L1Loss()(x, x)
    with pytest.raises(vlg_b200.VlgError):
        vlg_b200.warp(x, None, torch.zeros(1, 8, 8, 2))
    with pytest.raises(vlg_b200.VlgError):
        vlg_b200.ingest(torch.zeros(1, 8, 8, 3, dtype=torch.uint8))
    with pytest.raises(vlg_b200.VlgError):
        vlg_b200.warp_loss_labels(x, torch.zeros(1, 8, 8, dtype=torch.int64), torch.zeros(1, 8, 8, 2), x, torch.zeros(1, 8, 8, dtype=torch.int64))


def test_build_is_atomic_and_locked():
    """Every rank of a torchrun launch imports the package at once: the build must happen under a lock, into a
    temporary file that is moved into place (no rank may dlopen a half-written library)."""
    import inspect
    from vlg_b200 import _build
    src = inspect.getsource(_build.build_library)
    assert "flock" in src and "os.replace" in src
    assert not _build.is_stale(), "the in-tree library is older than its sources"


def test_product_never_imports_oracle():
    """The oracle is test infrastructure; the package must not import, load or execute it."""
    pkg = os.path.join(ROOT, "video-layout-generation_b200")
    pat = re.compile(r"import\s+oracle|from\s+oracle|from\s+\.+oracle|libvlg_oracle|c_oracle|torch_oracle|oracle/")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not pat.search(text), f
