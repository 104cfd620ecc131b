"""CPU-side checks of the C-ABI boundary: the shared library loads, exports every symbol that
include/dvd_b200.h declares, and the ctypes mirror of dvd_weights_t has the C layout.  No compute."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dvd_b200.h")


def _declared():
    txt = open(HEADER).read()
    return sorted(set(re.findall(r"DVD_API[^;(]*?\b(dvd_\w+)\s*\(", txt)))


def test_header_declares_entry_points():
    names = _declared()
    for must in ("dvd_unwarp_f32", "dvd_unwarp_u8", "dvd_sample", "dvd_denoise_step", "dvd_static_forward", "dvd_tables_init",
                 "dvd_workspace_bytes", "dvd_grid_sample_f32", "dvd_last_error", "dvd_version"):
        assert must in names


def test_library_exports_every_declared_symbol():
    from dvd_b200 import _lib
    lib = _lib.lib()
    for name in _declared():
        assert hasattr(lib, name), f"{name} declared in dvd_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in dvd_b200/_lib.py"
    assert lib.dvd_version() == 5
    assert lib.dvd_workspace_bytes(0, 2, 0) == 0
    assert lib.dvd_workspace_bytes(1, 2, 0) > 100 << 20


def test_ctypes_struct_layout_matches_c(tmp_path):
    """Compile a tiny C program against the header and compare sizeof/offsetof with the ctypes mirror."""
    from dvd_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvd_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(dvd_mat_t),sizeof(dvd_dec_layer_t),sizeof(dvd_weights_t),offsetof(dvd_weights_t,dec),'
                   'offsetof(dvd_weights_t,fin_ada_b),offsetof(dvd_dec_layer_t,conv2));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(_lib.Mat), C.sizeof(_lib.DecLayer), C.sizeof(_lib.Weights), _lib.Weights.dec.offset,
            _lib.Weights.fin_ada_b.offset, _lib.DecLayer.conv2.offset]
    assert got == want


def test_missing_library_fails_loudly(monkeypatch):
    from dvd_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libdvd_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()


def test_model_has_no_cpu_path():
    import torch
    from dvd_b200.model import DiT
    from oracle import synth
    m = DiT(precision="fp32")
    m.load_state_dict(synth.make_state_dict(1234, live_only=True), strict=False)
    assert next(m.parameters()).device.type == "cpu"
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(2, 2, 64, 64), torch.tensor([666.0, 666.0]), y512=torch.zeros(2, 3, 512, 512), mask_cat=torch.zeros(2, 1, 512, 512),
          mask_y512=torch.zeros(2, 384, 64, 64), line_msk=torch.zeros(2, 64, 64, 64), init_flow=torch.zeros(2, 2, 64, 64),
          init_feat=torch.zeros(2, 256, 64, 64), tv=True, iter=True)


def test_library_contains_blackwell_tensor_and_tma_instructions():
    """The shipped library is the hand-written sm_100a path: its SASS holds tcgen05.mma (UTCHMMA), TMEM loads (LDTM) and TMA
    loads / stores (UTMALDG / UTMASTG), and no legacy HMMA tensor instructions."""
    import shutil, subprocess
    from dvd_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump) or not os.path.exists(_lib.LIB_PATH):
        pytest.skip("cuobjdump or the built library is not available")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG", "UTMASTG"):
        assert mnemonic in sass, mnemonic
    assert " HMMA." not in sass and "HGMMA" not in sass
