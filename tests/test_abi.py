"""The C-ABI library loads on a CPU-only box and exports every symbol include/iefvad.h declares
(no compute calls here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "iefvad.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(iefvad_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from iefvad_b200 import _lib
    names = _declared()
    assert len(names) >= 10
    for n in names:
        assert hasattr(_lib.lib, n), f"{n} declared in include/iefvad.h but not exported by libiefvad.so"
    assert _lib.lib.iefvad_abi_version() == _lib.ABI_VERSION


def test_python_binding_covers_the_header():
    from iefvad_b200 import _lib
    assert set(_declared()) == set(_lib.EXPORTS)


def test_library_is_plain_c_abi_without_torch_dependency():
    import subprocess
    from iefvad_b200 import _lib
    r = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    # "name => path (0x<load address>)": the address is randomised per process and may spell "c10" - compare names
    # and paths only
    deps = [re.sub(r"\s*\(0x[0-9a-fA-F]+\)\s*$", "", line).strip() for line in r.stdout.splitlines() if line.strip()]
    assert any("libcudart" in d for d in deps), deps
    assert not any("torch" in d or "c10" in d for d in deps), deps


def test_invalid_arguments_fail_loudly_without_a_gpu():
    from iefvad_b200 import _lib
    h = ctypes.c_void_p()
    rc = _lib.lib.iefvad_model_create(h, 100, 8, 2, 10, 0.5, 1, 8.0, 1e-8)   # embed_dim not a multiple of 128
    assert rc != 0 and "embed_dim" in _lib.last_error()
    rc = _lib.lib.iefvad_model_create(h, 768, 7, 2, 10, 0.5, 1, 8.0, 1e-8)   # heads do not divide
    assert rc != 0 and "num_heads" in _lib.last_error()
