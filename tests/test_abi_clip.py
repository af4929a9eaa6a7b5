"""iefvad_clip_visual rejects malformed arguments before touching the device (runs without a GPU)."""
import ctypes as C


def _call(lib, N=2, dtype=1, R=224, P=14, W=1024, layers=2, heads=16, out_dim=768, plan=2, table=True):
    n = 8 + 12 * layers
    fake = (C.c_void_p * n)(*[256 * (i + 1) for i in range(n)])   # never dereferenced: every call below fails its checks
    return lib.iefvad_clip_visual(1 << 20, dtype, N, R, P, W, layers, heads, out_dim,
                                  C.cast(fake, C.c_void_p) if table else None, plan, 1 << 21, None)


def test_clip_visual_rejects_bad_arguments_without_a_gpu():
    from iefvad_b200 import _lib
    lib = _lib.lib
    for kwargs, text in (({"R": 230}, "multiple of patch"), ({"P": 0}, "multiple of patch"),
                         ({"W": 1000, "heads": 8}, "multiple of 128"), ({"W": 1152, "heads": 18}, "multiple of 128"),
                         ({"heads": 4}, "head dim 256"), ({"heads": 7}, "not divisible"),
                         ({"N": -1}, "outside [0, 65535]"), ({"N": 65536}, "outside [0, 65535]"),
                         ({"plan": 0}, "plan"), ({"plan": 1}, "plan"), ({"plan": 7}, "plan"),
                         ({"dtype": 3}, "dtype"), ({"dtype": -1}, "dtype"),
                         ({"table": False}, "null parameter table"), ({"layers": 65}, "layers"),
                         ({"out_dim": 0}, "output_dim")):
        assert _call(lib, **kwargs) != 0, kwargs
        assert text in _lib.last_error(), (kwargs, _lib.last_error())
