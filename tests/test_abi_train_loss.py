"""iefvad_train_loss_fwd / _bwd reject malformed arguments before touching the device (runs without a GPU)."""


def _fwd(lib, B=2, T=32, D=128, kmax=3, align=256, nu=8.0):
    p = [align * (i + 1) for i in range(16)]            # never dereferenced: every call below fails its argument checks
    return lib.iefvad_train_loss_fwd(p[0], p[1], 14, p[2], B, T, p[3], p[4], p[5], p[6], D, nu, 1.0, 1.0, p[7], p[8], kmax,
                                     p[9], p[10], p[11], p[12], p[13], None)


def test_train_loss_rejects_bad_arguments_without_a_gpu():
    from iefvad_b200 import _lib
    lib = _lib.lib
    for kwargs, text in (({"D": 6}, "D=6"), ({"kmax": 2}, "kmax"), ({"T": 0}, "out of range"), ({"align": 8}, "aligned"),
                         ({"nu": 0.0}, "nu")):
        assert _fwd(lib, **kwargs) != 0
        assert text in _lib.last_error(), (kwargs, _lib.last_error())
    rc = lib.iefvad_train_loss_bwd(256, 512, 768, 14, 1024, 2, 32, 3, 1280, 1536, 1792, 2048, 130, 2304, 8.0, 1.0, 1.0,
                                   None, None, None, None, 2560, 2816, 3072, 3328, 3584, None)
    assert rc != 0 and "D=130" in _lib.last_error()
