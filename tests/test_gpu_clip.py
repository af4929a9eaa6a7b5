"""CLIP VisionTransformer (extracting/clip/model.py:206-241) on the B200 vs the float64 torch port, at token counts
50 (attn_short), 257 and 577 (attn_long) and at full ViT-L/14 size."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import iefvad_oracle as O
from oracle import clip_visual as CV

pytestmark = pytest.mark.gpu

# (R, P, W, layers, heads, out_dim, N) -> tokens 50, 257, 577, and ViT-L/14 @ 224 (24 layers, 257 tokens)
SIZES = {"t50": (224, 32, 256, 2, 4, 128, 4), "t257": (224, 14, 256, 2, 4, 128, 4), "t577": (336, 14, 256, 2, 4, 128, 2),
         "vitl14": (224, 14, 1024, 24, 16, 768, 8)}
_CACHE = {}


def _case(name):
    """(module, x fp32 holding fp16-representable values, float64 reference, fp16 torch-port output)."""
    if name not in _CACHE:
        from iefvad_b200.clip import VisionTransformer
        R, P, W, layers, heads, out_dim, N = SIZES[name]
        sd = {k: torch.from_numpy(v) for k, v in CV.clip_visual_params(R, P, W, layers, out_dim, seed=3).items()}
        m = VisionTransformer(R, P, W, layers, heads, out_dim)
        m.load_state_dict(sd)
        m = m.cuda().eval().requires_grad_(False)
        g = torch.Generator("cpu").manual_seed(4)
        x = torch.randn((N, 3, R, R), generator=g).half().float().cuda()
        sd64 = {k: v.cuda() for k, v in sd.items()}
        with torch.no_grad():
            ref = CV.clip_visual_torch(x.double(), sd64, heads, torch.float64).cpu().numpy()
            ref16 = CV.clip_visual_torch(x, sd64, heads, torch.float16).float().cpu().numpy()
        del sd64
        _CACHE.clear()                      # keep one case resident (ViT-L's float64 weights are 2.4 GB)
        _CACHE[name] = (m, x, ref, ref16)
    return _CACHE[name]


def _run(m, x, precision):
    m.precision = precision
    with torch.no_grad():
        out = m(x)
    torch.cuda.synchronize()
    assert out.dtype == torch.float32 and out.shape == (x.shape[0], m.output_dim)
    return out


@pytest.mark.parametrize("name", list(SIZES))
def test_fp32_plan_vs_float64(name):
    """FFMA GEMMs and attention with fp32 LayerNorms.  Bound 1e-5 for every size; measured on one B200 (1000 W):
    7.4e-7 / 6.4e-7 / 8.0e-7 at 50 / 257 / 577 tokens, 1.8e-6 at ViT-L/14."""
    m, x, ref, _ = _case(name)
    err = O.max_norm_err(_run(m, x, "fp32").cpu().numpy(), ref)
    assert err < 1e-5, err


@pytest.mark.parametrize("name", list(SIZES))
def test_fp16_plan_no_worse_than_the_reference_fp16_arithmetic(name):
    """Default plan vs float64, bounded by the error of OpenAI's own fp16 forward (torch port in fp16 on the same
    GPU, same weights and inputs).  Measured on one B200 (1000 W), this path / torch fp16: 2.8e-4 / 8.5e-4 (50 tokens),
    3.3e-4 / 9.6e-4 (257), 4.0e-4 / 1.1e-3 (577), 6.7e-4 / 1.4e-3 (ViT-L/14)."""
    m, x, ref, ref16 = _case(name)
    err = O.max_norm_err(_run(m, x, "fp16").cpu().numpy(), ref)
    bar = O.max_norm_err(ref16, ref)
    assert err <= bar, (err, bar)


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_input_dtypes_give_identical_embeddings(precision):
    m, x, _, _ = _case("t257")
    x = (x * 32).round().clamp(-96, 96) / 32            # exact in fp16 and in bf16
    outs = [_run(m, x.to(dt), precision) for dt in (torch.float32, torch.float16, torch.bfloat16)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


@pytest.mark.parametrize("name,precision", [("vitl14", "fp16"), ("t50", "fp16"), ("t50", "fp32")])
def test_embedding_independent_of_the_batch(name, precision):
    m, x, _, _ = _case(name)
    g = torch.Generator("cpu").manual_seed(5)
    xb = torch.randn((64,) + tuple(x.shape[1:]), generator=g).half().float().cuda()
    big = _run(m, xb, precision)
    for i in (0, 1, 37, 63):
        assert torch.equal(_run(m, xb[i:i + 1], precision)[0], big[i]), i


def test_grad_enabled_and_cpu_inputs_raise():
    from iefvad_b200.clip import VisionTransformer
    m = VisionTransformer(28, 14, 128, 1, 2, 64).cuda()
    x = torch.randn(2, 3, 28, 28, device="cuda")
    with pytest.raises(RuntimeError, match="no_grad"):
        m(x)                                            # parameters require grad
    m.requires_grad_(False)
    with pytest.raises(RuntimeError, match="no_grad"):
        m(x.clone().requires_grad_(True))
    with torch.no_grad():
        assert m(x).shape == (2, 64)
        with pytest.raises(RuntimeError, match="CUDA"):
            m(x.cpu())
        with pytest.raises(RuntimeError, match=r"\[N, 3, 28, 28\]"):
            m(x[:, :, :14])
        m.precision = "bf16"
        with pytest.raises(RuntimeError, match="plan"):
            m(x)


def test_module_transformer_fp16_plan_vs_reference_golden():
    """The fp16 plan on the D4 path (masked attention, key padding).  Bound 1e-3 (the bf16 plan's is 3e-2); measured
    on one B200 (1000 W): 1.8e-4 with the mask and key padding, 1.6e-4 with the mask only."""
    from iefvad_b200 import module
    z = load_golden("layers.npz")
    c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    W, heads = z["tr:x"].shape[-1], int(z["tr:heads"])
    layers_n = len({k.split(".")[1] for k in z.files if k.startswith("tr:param:resblocks.")})
    tr = module.Transformer(W, layers_n, heads, attn_mask=c(z["tr:mask"])).cuda().eval()
    tr.load_state_dict({k[len("tr:param:"):]: c(z[k]) for k in z.files if k.startswith("tr:param:")})
    tr.precision = "fp16"
    out_m, _ = tr((c(z["tr:x"]), c(z["tr:pad"])))
    out_p, _ = tr((c(z["tr:x"]), None))
    assert O.max_norm_err(out_m.cpu().numpy(), z["tr:out_masked"]) < 1e-3
    assert O.max_norm_err(out_p.cpu().numpy(), z["tr:out_nopad"]) < 1e-3
