"""The model's precision plans: HH (default), B and fp32 are accepted; every other plan code or name is rejected
without changing the model."""
import pytest
import torch

REMOVED_CODES = (0, 2, 7, 10, 26, 57, 64)


@pytest.mark.gpu
def test_set_plan_accepts_hh_b_fp32_and_rejects_other_codes():
    assert torch.cuda.is_available()
    from iefvad_b200 import _lib
    h = _lib._vp()
    _lib.check(_lib.lib.iefvad_model_create(h, 128, 4, 1, 1, 0.5, 0, 5.0, 1e-8))
    try:
        assert _lib.lib.iefvad_model_get_plan(h.value) == _lib.PLANS["HH"] == 56
        for plan in (-1, 6, 56):
            _lib.check(_lib.lib.iefvad_model_set_plan(h.value, plan))
            assert _lib.lib.iefvad_model_get_plan(h.value) == plan
            for bad in REMOVED_CODES:
                assert _lib.lib.iefvad_model_set_plan(h.value, bad) == 1          # IEFVAD_ERR_INVALID
                msg = _lib.last_error()
                assert f"plan {bad}" in msg and all(s in msg for s in ("HH (56)", "B (6)", "FP32 (-1)")), msg
                assert _lib.lib.iefvad_model_get_plan(h.value) == plan
    finally:
        _lib.lib.iefvad_model_destroy(h.value)


@pytest.mark.parametrize("name", ["A", "H", "H8", "bf16", "split"])
def test_removed_plan_name_raises_before_any_device_call(name):
    import iefvad_b200
    from iefvad_b200 import synth
    m = iefvad_b200.MMFMIL(14, 128, 256, 128, 4, 1, 8, 10, 10, "cuda:0",
                           synth.default_args(visual_layers=1, visual_head=4, num_refinement_steps=1))
    m.temporal.precision = name
    x = torch.zeros(1, 8, 128, dtype=torch.float16)
    with pytest.raises(ValueError, match=r"choose from \['B', 'HH', 'fp32'\]"):
        m.temporal.scores(x, x, device="cuda:0")
    assert m.temporal._handle is None
