// CLIP image encoder of the feature-extraction step (SURVEY row N4): OpenAI's VisionTransformer,
// extracting/clip/model.py:206-241, on the GEMM / attention / LayerNorm kernels of the D4 transformer.
#pragma once
#include "common.cuh"
#include "graph.cuh"

namespace iefvad {

struct ClipVisualParams {   // fp32 device pointers, the layout of VisionTransformer.state_dict()
  const float* conv1;       // [width, 3, P, P]
  const float* cls;         // class_embedding [width]
  const float* pos;         // positional_embedding [G*G + 1, width]
  const float *ln_pre_w, *ln_pre_b;
  const ResBlockParams* blocks;   // [layers]
  const float *ln_post_w, *ln_post_b;
  const float* proj;        // [width, output_dim]
};

// x [N, 3, R, R] (dtype IEFVAD_DT_F32 / F16 / BF16, normalised pixels) -> out [N, output_dim] fp32.
// plan: -1 fp32 FFMA, 2 fp16 operands (fp32 accumulation, LayerNorm and residual).  Validates every argument before
// touching the device.
int clip_visual(const void* x, int dtype, int N, int resolution, int patch, int width, int layers, int heads,
                int output_dim, const ClipVisualParams& p, int plan, float* out, cudaStream_t stream);

}  // namespace iefvad
