"""CLIP VisionTransformer (extracting/clip/model.py:206-241): the numpy oracle, the float64 torch port and the
independent `transformers` implementation agree; `VisionTransformer.from_state_dict` infers OpenAI's configuration.
Runs without a GPU."""
import numpy as np
import pytest
import torch

from oracle import iefvad_oracle as O
from oracle import clip_visual as CV

# (R, P, W, layers, heads, out_dim, N): a 5-token toy, and a ViT-B/32-shaped one with 50 tokens
CONFIGS = [(28, 14, 128, 2, 2, 64, 3), (224, 32, 768, 1, 12, 512, 2)]


def _inputs(R, P, W, layers, out_dim, N, seed=0):
    sd = CV.clip_visual_params(R, P, W, layers, out_dim, seed)
    x = np.random.default_rng(seed + 1).standard_normal((N, 3, R, R))
    return sd, x


def _hf_model(sd, R, P, W, layers, heads, out_dim):
    tr = pytest.importorskip("transformers")
    cfg = tr.CLIPVisionConfig(hidden_size=W, intermediate_size=4 * W, num_hidden_layers=layers, num_attention_heads=heads,
                              image_size=R, patch_size=P, hidden_act="quick_gelu", projection_dim=out_dim,
                              layer_norm_eps=1e-5)
    m = tr.CLIPVisionModelWithProjection(cfg).double().eval()
    t = {k: torch.from_numpy(v) for k, v in sd.items()}
    hf = {"vision_model.embeddings.class_embedding": t["class_embedding"],
          "vision_model.embeddings.patch_embedding.weight": t["conv1.weight"],
          "vision_model.embeddings.position_embedding.weight": t["positional_embedding"],
          "vision_model.pre_layrnorm.weight": t["ln_pre.weight"], "vision_model.pre_layrnorm.bias": t["ln_pre.bias"],
          "vision_model.post_layernorm.weight": t["ln_post.weight"], "vision_model.post_layernorm.bias": t["ln_post.bias"],
          "visual_projection.weight": t["proj"].T.contiguous()}
    for i in range(layers):
        src, dst = f"transformer.resblocks.{i}.", f"vision_model.encoder.layers.{i}."
        for j, qkv in enumerate("qkv"):
            hf[dst + f"self_attn.{qkv}_proj.weight"] = t[src + "attn.in_proj_weight"][j * W:(j + 1) * W]
            hf[dst + f"self_attn.{qkv}_proj.bias"] = t[src + "attn.in_proj_bias"][j * W:(j + 1) * W]
        for a, b in (("attn.out_proj", "self_attn.out_proj"), ("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"),
                     ("mlp.c_fc", "mlp.fc1"), ("mlp.c_proj", "mlp.fc2")):
            hf[dst + b + ".weight"] = t[src + a + ".weight"]
            hf[dst + b + ".bias"] = t[src + a + ".bias"]
    missing, unexpected = m.load_state_dict(hf, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    return m


@pytest.mark.parametrize("R,P,W,layers,heads,out_dim,N", CONFIGS)
def test_oracle_torch_port_and_transformers_agree_in_float64(R, P, W, layers, heads, out_dim, N):
    sd, x = _inputs(R, P, W, layers, out_dim, N)
    ref = CV.clip_visual(x, sd, heads)
    assert ref.shape == (N, out_dim) and np.all(np.isfinite(ref))
    port = CV.clip_visual_torch(torch.from_numpy(x), {k: torch.from_numpy(v) for k, v in sd.items()}, heads, torch.float64)
    assert O.max_norm_err(port.numpy(), ref) < 1e-10
    m = _hf_model(sd, R, P, W, layers, heads, out_dim)
    with torch.no_grad():
        hf = m(pixel_values=torch.from_numpy(x)).image_embeds
    assert O.max_norm_err(hf.numpy(), ref) < 1e-10


def test_torch_port_fp16_follows_the_fp32_forward():
    """The fp16 arm is OpenAI's fp16 arithmetic: close to float64, not equal (checked on CPU in float32 here; the fp16
    arm itself runs on CUDA in tests/test_gpu_clip.py)."""
    R, P, W, layers, heads, out_dim, N = CONFIGS[0]
    sd, x = _inputs(R, P, W, layers, out_dim, N)
    ref = CV.clip_visual(x, sd, heads)
    f32 = CV.clip_visual_torch(torch.from_numpy(x), {k: torch.from_numpy(v) for k, v in sd.items()}, heads, torch.float32)
    assert f32.dtype == torch.float32
    assert O.max_norm_err(f32.numpy(), ref) < 1e-5


def test_from_state_dict_infers_vit_l14_from_an_fp16_checkpoint():
    from iefvad_b200.clip import VisionTransformer
    W, layers, P, G, out_dim = 1024, 24, 14, 16, 768
    shapes = {"conv1.weight": (W, 3, P, P), "class_embedding": (W,), "positional_embedding": (G * G + 1, W),
              "ln_pre.weight": (W,), "ln_pre.bias": (W,), "ln_post.weight": (W,), "ln_post.bias": (W,),
              "proj": (W, out_dim)}
    for i in range(layers):
        pre = f"transformer.resblocks.{i}."
        shapes.update({pre + "ln_1.weight": (W,), pre + "ln_1.bias": (W,), pre + "attn.in_proj_weight": (3 * W, W),
                       pre + "attn.in_proj_bias": (3 * W,), pre + "attn.out_proj.weight": (W, W),
                       pre + "attn.out_proj.bias": (W,), pre + "ln_2.weight": (W,), pre + "ln_2.bias": (W,),
                       pre + "mlp.c_fc.weight": (4 * W, W), pre + "mlp.c_fc.bias": (4 * W,),
                       pre + "mlp.c_proj.weight": (W, 4 * W), pre + "mlp.c_proj.bias": (W,)})
    # a distinct fp16 value per tensor (exact in fp32), so that every load is visible
    sd = {k: torch.full(s, (j % 97 - 48) / 64.0, dtype=torch.float16) for j, (k, s) in enumerate(shapes.items())}
    m = VisionTransformer.from_state_dict(sd)
    assert (m.input_resolution, m.conv1.kernel_size[0], m.conv1.out_channels, m.transformer.layers, m.heads,
            m.output_dim) == (224, 14, 1024, 24, 16, 768)
    got = m.state_dict()
    assert set(got) == set(sd)
    for k, v in sd.items():
        assert got[k].dtype == torch.float32 and torch.equal(got[k], v.float()), k
    assert m.precision == "fp16"
