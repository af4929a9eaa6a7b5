"""tcgen05 GEMM micro-benchmark of single epilogue kinds: python scripts/bench_gemm_epi.py M kind [kind ...]"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iefvad_b200 import _lib  # noqa: E402

M = int(sys.argv[1])
for epi in [int(x) for x in sys.argv[2:]]:
    ms = C.c_float()
    _lib.check(_lib.lib.iefvad_bench_gemm(M, 768, 768, 1, 512, 0, epi, 30, C.byref(ms)))
    print(f"M={M} epi_kind={epi}: {ms.value * 1e3:.1f} us  "
          f"{2.0 * M * 768 * 768 / ms.value / 1e9:.0f} TF/s", flush=True)
