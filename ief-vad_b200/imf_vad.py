"""Drop-in replacements for the reference's `model.imf_vad.MMFMIL` and `MultiModal_Fusion_Attn_Iter`
(model/imf_vad.py:5-161) whose forward runs entirely in libiefvad.so on an sm_100a GPU.

Same constructor signatures, attributes, `forward(img_visual, ev_visual, padding_mask, text, lengths,
return_attn=False)` signature, output dict (8 fp32 tensors, model/imf_vad.py:152-161) and `state_dict()` keys /
shapes, so `main.py`, `test.py`, `test2.py` and `train/*_test.py` of the reference can use it unchanged (see
INTEGRATION.md for the one-line shim).  The nn.Module only *owns* the parameters (fp32 `nn.Parameter`s, created
in the reference's order so `torch.manual_seed(s)` yields bit-identical initial weights); all arithmetic happens
in hand-written CUDA kernels reached through the C ABI - there is no PyTorch or CPU fallback."""
from __future__ import annotations

import os
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib

_MODALITIES = ("image", "event")
_DTYPE_CODES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}


def _norm_device(device) -> torch.device:
    """torch.device with an explicit index ("cuda" -> "cuda:<current>"), so it compares equal to tensor.device."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class MultiModal_Fusion_Attn_Iter(nn.Module):
    """Parameter layout of model/imf_vad.py:69-107; forward of :109-161 on the GPU."""

    def __init__(self, embed_dim, num_layers=2, num_heads=8, dropout=0.1, num_refinement_steps=3, lambda_ref=0.5,
                 noise_model="StudentT", nu=5, epsilon=1e-8):
        super().__init__()
        self.embed_dim = embed_dim
        self.num_layers = num_layers
        self.num_heads = num_heads
        self.num_refinement_steps = num_refinement_steps
        self.lambda_ref = lambda_ref
        self.noise_model = noise_model
        self.nu = nu
        self.epsilon = epsilon
        self.dropout = dropout          # attention dropout only acts in train(); this path is forward-only (eval)
        # mask of the train() attention dropout: "philox" = the library's own counter-based mask, seeded from torch's CPU
        # generator; "torch" = PyTorch's own mask, drawn from (and advancing) the device's CUDA generator exactly like
        # nn.MultiheadAttention does, so a seeded run sees the reference's masks and random streams (include/iefvad.h)
        self.dropout_rng = "philox"
        self.precision = os.environ.get("IEFVAD_PLAN", "HH")
        # valid-rows evaluation forward: compute the identical zero-pad rows of a chunk once (DESIGN.md, pad de-duplication)
        self.pad_dedup = True
        # refinement chain as one persistent kernel: None = when the batch is large enough (library default), False /
        # True = never / always (both forms produce identical bits; iefvad_model_set_option "refine_fused")
        self.refine_fused = None
        # fused encoder tails / heads (csrc/outproj_ln.cu, heads_fuse.cu); False = the separate GEMM + row-wise launches
        self.outproj_ln = True
        self.heads_fuse = True
        # range guard of the 16-bit plans: "raise" (default) = check_finite() / Evaluator.finish() raise when a forward
        # produced a non-finite logit; "fallback" = the Evaluator re-runs the pass under the bf16 plan "B"
        self.on_overflow = os.environ.get("IEFVAD_ON_OVERFLOW", "raise")
        self.check_every_forward = os.environ.get("IEFVAD_CHECK", "0") not in ("", "0")

        # nn.MultiheadAttention / LayerNorm / Linear instances are used purely as parameter containers: they give
        # the reference's state_dict keys and consume the RNG exactly like the reference constructor does
        # (attention stacks of both modalities first, then the four heads, the refinement MLPs, the classifier).
        for mod in _MODALITIES:
            setattr(self, f"{mod}_attn_layers", nn.ModuleList(
                nn.MultiheadAttention(embed_dim, num_heads, dropout=dropout, batch_first=True)
                for _ in range(num_layers)))
            setattr(self, f"{mod}_norms", nn.ModuleList(nn.LayerNorm(embed_dim) for _ in range(num_layers)))
        for mod in _MODALITIES:
            setattr(self, f"whiten_{mod}", nn.LayerNorm(embed_dim))
        for kind in ("mu", "logvar"):
            for mod in _MODALITIES:
                setattr(self, f"{mod}_{kind}", nn.Linear(embed_dim, embed_dim))
        if num_refinement_steps == 0:
            blocks = [nn.Identity()]
        else:
            blocks = [nn.Sequential(nn.Linear(embed_dim, embed_dim), nn.ReLU(), nn.Linear(embed_dim, embed_dim))
                      for _ in range(num_refinement_steps)]
        self.refinement_blocks = nn.ModuleList(blocks)
        self.classifier = nn.Linear(embed_dim, 1)

        self._handle: Optional[int] = None
        self._handle_device: Optional[torch.device] = None
        self._uploaded: Dict[str, tuple] = {}

    # ------------------------------------------------------------------ native model management
    def _release(self):
        self.__dict__.pop("_graphs", None)       # captured graphs hold addresses of the handle's workspaces
        if getattr(self, "_handle", None):
            _lib.lib.iefvad_model_destroy(self._handle)
        self._handle = None
        self._uploaded = {}

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _native(self, device: torch.device) -> int:
        if self._handle is not None and self._handle_device == device:
            return self._handle
        self._release()
        if self.noise_model not in _lib.NOISE:                       # model/imf_vad.py:137-138
            raise ValueError("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'.")
        h = _lib._vp()
        with torch.cuda.device(device):
            _lib.check(_lib.lib.iefvad_model_create(
                h, int(self.embed_dim), int(self.num_heads), int(self.num_layers), int(self.num_refinement_steps),
                float(self.lambda_ref), _lib.NOISE[self.noise_model], float(self.nu), float(self.epsilon)))
        self._handle, self._handle_device = h.value, device
        max_rows = int(os.environ.get("IEFVAD_MAX_ROWS", "0") or 0)          # rows per internal slab (tuning knob)
        if max_rows > 0:
            _lib.check(_lib.lib.iefvad_model_set_max_rows(self._handle, max_rows))
        return self._handle

    def refresh_weights(self) -> None:
        """Force a re-upload of every parameter on the next forward.  The automatic check compares (storage address,
        tensor version) per parameter, which sees load_state_dict, optimizer steps, .to() and every in-place op on the
        parameter itself - but NOT writes through `.data` (p.data.mul_(), EMA updates on .data), which bypass the
        version counter: call this after such an update."""
        self._uploaded = {}

    def check_finite(self) -> bool:
        """Range guard (synchronises): True when every logit produced since the last check was finite.  fp16 operands
        saturate at 65 504 where the reference's fp32 does not; an overflow anywhere upstream reaches the classifier
        as inf / NaN and sets a device flag (include/iefvad.h, iefvad_model_check_finite)."""
        if self._handle is None:
            return True
        import ctypes as C
        flag = C.c_int(0)
        with torch.cuda.device(self._handle_device):
            _lib.check(_lib.lib.iefvad_model_check_finite(self._handle, C.byref(flag),
                                                          torch.cuda.current_stream(self._handle_device).cuda_stream))
        if flag.value & 2:
            raise RuntimeError("pad de-duplication needs the valid rows of every chunk to be its FIRST rows: the row map passed "
                               "to scores() is not the prefix map; set model.temporal.pad_dedup = False for other maps")
        return flag.value == 0

    def _raise_overflow(self):
        raise FloatingPointError(
            f"IEF-VAD B200 path: precision plan {self.precision!r} produced non-finite logits - a 16-bit operand left "
            "the fp16 range (65 504).  Re-run with model.temporal.precision = 'B' (bf16 operands, fp32's exponent range) "
            "or 'fp32'.")

    def _set_eval_outputs(self, h: int, extra: Optional[Dict[str, torch.Tensor]], n_rows: int, device) -> None:
        """Register (or clear, extra=None) the optional outputs of the evaluation forward: what the reference's loop
        derives per frame besides the score (train/ucf_test.py:124-144).  Keys: "wi_mean", "we_mean" [rows] and
        "fused", "image_mu", "event_mu" [rows, D] - fp32 device tensors of the caller (compact in valid-rows mode)."""
        ptrs = [0] * 5
        if extra:
            for i, (key, width) in enumerate((("wi_mean", 1), ("we_mean", 1), ("fused", self.embed_dim),
                                              ("image_mu", self.embed_dim), ("event_mu", self.embed_dim))):
                t = extra.get(key)
                if t is None:
                    continue
                if (not t.is_cuda or t.device != device or t.dtype != torch.float32 or not t.is_contiguous()
                        or t.numel() != n_rows * width):
                    raise RuntimeError(f"extra output {key!r} must be a contiguous fp32 tensor of {n_rows * width} "
                                       f"elements on {device}")
                ptrs[i] = t.data_ptr()
            unknown = set(extra) - {"wi_mean", "we_mean", "fused", "image_mu", "event_mu"}
            if unknown:
                raise KeyError(f"unknown extra outputs {sorted(unknown)}")
        _lib.check(_lib.lib.iefvad_model_set_eval_outputs(h, *ptrs))

    def _apply_options(self, h: int) -> None:
        mode = -1 if self.refine_fused is None else (int(self.refine_fused) if not isinstance(self.refine_fused, bool)
                                                     else int(self.refine_fused))
        _lib.check(_lib.lib.iefvad_model_set_option(h, b"refine_fused", mode))
        _lib.check(_lib.lib.iefvad_model_set_option(h, b"outproj_ln", int(bool(self.outproj_ln))))
        _lib.check(_lib.lib.iefvad_model_set_option(h, b"heads_fuse", int(bool(self.heads_fuse))))

    def _sync_params(self, handle: int, device: torch.device, stream: int) -> None:
        """Upload parameters whose storage or version changed since the last forward (load_state_dict,
        optimizer steps, .to(), in-place ops on the parameter); see `refresh_weights` for writes through `.data`."""
        self._apply_options(handle)
        for name, p in self.named_parameters():
            tag = (p.data_ptr(), p._version)
            if self._uploaded.get(name) == tag:
                continue
            if p.device != device:
                raise RuntimeError(f"parameter {name} is on {p.device} but the inputs are on {device}; "
                                   "call model.to(device) first")
            src = p.detach()
            if src.dtype != torch.float32 or not src.is_contiguous():
                src = src.float().contiguous()
            _lib.check(_lib.lib.iefvad_model_set_param(handle, ("temporal." + name).encode(), src.data_ptr(),
                                                       src.numel(), stream))
            self._uploaded[name] = tag

    def _prepare(self, device: torch.device) -> Tuple[int, int]:
        """The native model on `device` with current parameters, options, precision plan and pad de-duplication:
        (handle, stream).  An unknown plan name raises ValueError before anything touches the device."""
        plan = _lib.PLANS.get(str(self.precision))
        if plan is None:
            raise ValueError(f"unknown precision plan {self.precision!r}; choose from {sorted(_lib.PLANS)}")
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            h = self._native(device)
            self._sync_params(h, device, stream)
            _lib.check(_lib.lib.iefvad_model_set_plan(h, plan))
            _lib.check(_lib.lib.iefvad_model_set_pad_dedup(h, 1 if self.pad_dedup else 0))
        return h, stream

    # ------------------------------------------------------------------ forward
    def forward(self, image_features: torch.Tensor, event_features: torch.Tensor,
                with_scores: bool = False) -> Dict[str, torch.Tensor]:
        if self.noise_model not in _lib.NOISE:
            raise ValueError("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'.")
        if self.dropout_rng not in _lib.DROPOUT_KINDS:
            raise ValueError(f"unknown dropout_rng {self.dropout_rng!r}; choose from {sorted(_lib.DROPOUT_KINDS)}")
        if not (image_features.is_cuda and event_features.is_cuda):
            raise RuntimeError("IEF-VAD B200 path is CUDA-only: inputs must live on an sm_100a device "
                               "(there is no CPU fallback)")
        needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                                  or image_features.requires_grad or event_features.requires_grad)
        if needs_grad or (self.training and self.dropout > 0):
            # training step (row N3): autograd node over the library's kernels; attention dropout in train() mode
            return self._forward_train(image_features, event_features)
        if image_features.dim() != 3 or image_features.shape != event_features.shape:
            raise RuntimeError(f"expected two [B, T, {self.embed_dim}] tensors, got {tuple(image_features.shape)} "
                               f"and {tuple(event_features.shape)}")
        B, T, D = image_features.shape
        if D != self.embed_dim:
            raise RuntimeError(f"last dimension {D} != embed_dim {self.embed_dim}")
        device = image_features.device
        if image_features.dtype not in _DTYPE_CODES or event_features.dtype != image_features.dtype:
            image_features, event_features = image_features.float(), event_features.float()
        img = image_features.contiguous()
        ev = event_features.contiguous()
        h, _ = self._prepare(device)
        with torch.cuda.device(device):
            def launch(img_t, ev_t, wide_t, logits_t, scores_t):
                _lib.check(_lib.lib.iefvad_model_forward(
                    h, img_t.data_ptr(), ev_t.data_ptr(), _DTYPE_CODES[img_t.dtype], B, T,
                    wide_t[0].data_ptr(), logits_t.data_ptr(), wide_t[1].data_ptr(), wide_t[2].data_ptr(),
                    wide_t[3].data_ptr(), wide_t[4].data_ptr(), wide_t[5].data_ptr(), wide_t[6].data_ptr(),
                    _lib.ptr(scores_t), torch.cuda.current_stream(device).cuda_stream))

            # Small problems are bound by launching ~60 kernels from the host (0.5 ms for one 256-row clip): replay
            # them as one CUDA graph over static buffers (two copies in, one clone out).  IEFVAD_GRAPH_ROWS=0 disables.
            replay = self._graph_replay(device, B, T, D, img, ev, with_scores, launch) if B * T else None
            if replay is not None:
                wide, logits, scores = replay
            else:
                wide = torch.empty((7, B, T, D), dtype=torch.float32, device=device)
                logits = torch.empty((B, T, 1), dtype=torch.float32, device=device)
                scores = torch.empty((B, T), dtype=torch.float32, device=device) if with_scores else None
                launch(img, ev, wide, logits, scores)
        if self.check_every_forward and not self.check_finite():
            self._raise_overflow()
        out = {
            "fused": wide[0], "logits": logits, "image_mu": wide[1], "event_mu": wide[2],
            "image_logvar": wide[3], "event_logvar": wide[4], "w_i": wide[5], "w_e": wide[6],
        }
        if with_scores:
            out["scores"] = scores
        return out


    def _forward_train(self, image_features: torch.Tensor, event_features: torch.Tensor) -> Dict[str, torch.Tensor]:
        """model/imf_vad.py:109-161 with a grad_fn (train.ForwardFn): what `loss.backward()` of train/ucf_train.py:105 needs.
        Attention dropout (p = self.dropout) is applied in train() mode only, like nn.MultiheadAttention.  dropout_rng
        "philox": every call draws a fresh Philox seed from torch's CPU generator, so `torch.manual_seed` makes runs
        reproducible.  "torch": the CPU generator is left alone; the four attention layers take torch.native_dropout's
        masks at consecutive offsets of the device's CUDA generator (image L0, L1, event L0, L1, the reference's order),
        which is then advanced past them - the masks and every later CUDA draw are the reference's."""
        from . import train
        if image_features.dim() != 3 or image_features.shape != event_features.shape or image_features.shape[-1] != self.embed_dim:
            raise RuntimeError(f"expected two [B, T, {self.embed_dim}] tensors, got {tuple(image_features.shape)} "
                               f"and {tuple(event_features.shape)}")
        p_drop = float(self.dropout) if self.training else 0.0
        B, T = int(image_features.shape[0]), int(image_features.shape[1])
        seed, offsets, threads = 0, None, 0
        if p_drop > 0 and self.dropout_rng == "torch" and B * T > 0:
            seed, offsets, threads = self._torch_dropout_state(image_features.device, B * self.num_heads * T * T)
        elif p_drop > 0:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        cfg = dict(layers=self.num_layers, steps=self.num_refinement_steps, heads=self.num_heads, p_drop=p_drop, seed=seed,
                   offsets=offsets, threads=threads, lambda_ref=float(self.lambda_ref), noise_model=self.noise_model,
                   nu=float(self.nu), epsilon=float(self.epsilon))
        outs = train.ForwardFn.apply(cfg, image_features, event_features, *train.param_list(self))
        keys = ("fused", "logits", "image_mu", "event_mu", "image_logvar", "event_logvar", "w_i", "w_e")
        return dict(zip(keys, outs))

    def _torch_dropout_state(self, device: torch.device, n: int):
        """(seed, per-layer offsets, launch width) of torch.native_dropout on the n = B*H*T*T attention weights of each
        layer, read from the CUDA generator of `device`, which is advanced past all of them as the reference's forward
        would advance it."""
        from . import ops
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("dropout_rng = 'torch' reads and advances the CUDA generator on the host, which CUDA-graph "
                               "capture does not support; capture with dropout_rng = 'philox' or in eval() mode")
        if n % 4:
            raise RuntimeError(f"dropout_rng = 'torch' needs B*heads*T*T to be a multiple of 4 (got {n}): torch draws other "
                               "sizes with a narrower vector width, which the kernels do not reproduce")
        torch.cuda.init()                                           # default_generators is filled on initialisation
        index = device.index if device.index is not None else torch.cuda.current_device()
        gen = torch.cuda.default_generators[index]
        threads, advance = ops.torch_dropout_launch(n, index)
        seed, offset = int(gen.initial_seed()), int(gen.get_offset())
        layers = 2 * self.num_layers                                # image L0 .. L-1, then event L0 .. L-1
        gen.set_offset(offset + layers * advance)
        return seed, [offset + k * advance for k in range(layers)], threads

    def _graph_replay(self, device, B, T, D, img, ev, with_scores, launch):
        """One CUDA-graph replay of the forward for a small [B, T] problem, or None (too large, disabled, already
        capturing, or capture failed once for this shape).  The graph is captured over static input / output buffers
        after an eager warm-up call that sizes every library workspace; parameters live in the library's own arena, so
        a `load_state_dict` / optimizer step between calls is picked up by the replay."""
        limit = int(os.environ.get("IEFVAD_GRAPH_ROWS", "2048") or 0)
        if B * T > limit or torch.cuda.is_current_stream_capturing():
            return None
        key = (str(device), B, T, img.dtype, str(self.precision), bool(with_scores), self.refine_fused, self.outproj_ln,
               self.heads_fuse)
        cache = self.__dict__.setdefault("_graphs", {})
        entry = cache.get(key)
        if entry is False:
            return None
        if entry is not None and entry[4] != _lib.lib.iefvad_alloc_generation():
            entry = None                        # a larger call re-allocated a workspace since the capture
        n_wide = 7 * B * T * D
        if entry is None:
            try:
                s_img, s_ev = torch.empty_like(img), torch.empty_like(ev)
                s_out = torch.empty(n_wide + 2 * B * T, dtype=torch.float32, device=device)
                wide = s_out[:n_wide].view(7, B, T, D)
                logits = s_out[n_wide:n_wide + B * T].view(B, T, 1)
                scores = s_out[n_wide + B * T:].view(B, T) if with_scores else None
                s_img.copy_(img)
                s_ev.copy_(ev)
                side = torch.cuda.Stream(device)
                side.wait_stream(torch.cuda.current_stream(device))
                with torch.cuda.stream(side):
                    launch(s_img, s_ev, wide, logits, scores)            # sizes the workspaces outside the capture
                torch.cuda.current_stream(device).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                l0 = _lib.lib.iefvad_launch_count()
                with torch.cuda.graph(graph):
                    launch(s_img, s_ev, wide, logits, scores)
                n_kernels = _lib.lib.iefvad_launch_count() - l0
                if len(cache) >= 4:                                      # a handful of shapes; drop the oldest
                    cache.pop(next(iter(cache)))
                entry = cache[key] = (graph, s_img, s_ev, s_out, _lib.lib.iefvad_alloc_generation(), n_kernels)
            except Exception:
                cache[key] = False
                return None
        graph, s_img, s_ev, s_out, _, n_kernels = entry
        s_img.copy_(img)
        s_ev.copy_(ev)
        graph.replay()
        _lib.lib.iefvad_add_launches(n_kernels)
        out = s_out.clone()
        return (out[:n_wide].view(7, B, T, D), out[n_wide:n_wide + B * T].view(B, T, 1),
                out[n_wide + B * T:].view(B, T) if with_scores else None)

    def scores(self, img: torch.Tensor, ev: torch.Tensor, device=None, valid_lengths=None, rowmap=None,
               extra: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """Evaluation forward (iefvad_model_forward_scores): device `logits` / `scores` only.

        img / ev: [B, T, D] on the device, or on the HOST (ideally pinned; `device` then names the GPU) - host inputs
        go through the library's pipelined copy (part p+1 travels while part p computes); nothing waits for the device,
        so host tensors must stay alive and unchanged until the stream has run.
        valid_lengths (host int64 [B]) + rowmap (device int32 [sum len], b * T + t of every valid row): the "valid rows"
        mode for zero-padded chunks - stages after the last attention core run on the valid rows only and the results
        are COMPACT [sum len]: bit-identical to the valid rows of the full forward with `pad_dedup = False`, within
        the rounding of one softmax term of them with the default pad de-duplication (rows past the valid length are
        then taken to be the zero pads of `process_split` and are not read)."""
        if img.dim() != 3 or img.shape != ev.shape or img.shape[-1] != self.embed_dim:
            raise RuntimeError(f"expected two [B, T, {self.embed_dim}] tensors")
        if img.dtype not in _DTYPE_CODES or ev.dtype != img.dtype:
            raise RuntimeError("inputs must share one of the dtypes float32 / float16 / bfloat16")
        on_host = not img.is_cuda
        if on_host != (not ev.is_cuda):
            raise RuntimeError("img and ev must both be on the host or both on the device")
        device = _norm_device(device) if on_host else img.device
        if on_host and device.type != "cuda":
            raise RuntimeError("host inputs need the target CUDA device")
        img, ev = img.contiguous(), ev.contiguous()
        B, T, _ = img.shape
        if (valid_lengths is None) != (rowmap is None):
            raise RuntimeError("valid_lengths and rowmap go together")
        n_out, lens_ptr, keep = B * T, None, (img, ev)
        if valid_lengths is not None:
            import ctypes as C
            lens = [int(v) for v in valid_lengths]
            if len(lens) != B or rowmap.dtype != torch.int32 or not rowmap.is_cuda or rowmap.numel() != sum(lens):
                raise RuntimeError("valid_lengths must have B entries and rowmap must be a device int32 tensor of sum(len)")
            arr = (C.c_int64 * B)(*lens)
            lens_ptr, n_out, keep = C.cast(arr, C.c_void_p), sum(lens), (img, ev, arr, rowmap)
        h, stream = self._prepare(device)
        with torch.cuda.device(device):
            logits = torch.empty(max(n_out, 1), dtype=torch.float32, device=device)[:n_out]
            scores = torch.empty(max(n_out, 1), dtype=torch.float32, device=device)[:n_out]
            self._set_eval_outputs(h, extra, n_out, device)
            try:
                _lib.check(_lib.lib.iefvad_model_forward_scores(
                    h, img.data_ptr(), ev.data_ptr(), _DTYPE_CODES[img.dtype], int(on_host), B, T, lens_ptr, _lib.ptr(rowmap),
                    logits.data_ptr(), scores.data_ptr(), stream))
            finally:
                if extra:
                    self._set_eval_outputs(h, None, 0, device)
        if valid_lengths is None:
            logits, scores = logits.view(B, T, 1), scores.view(B, T)
        return {"logits": logits, "scores": scores, "_keepalive": keep}

    def scores_ragged(self, img_packed: torch.Tensor, ev_packed: torch.Tensor, device, T: int, valid_lengths, rowmap,
                      chunk_start, chunk_valid, extra: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """Evaluation forward from RAGGED host features (iefvad_model_forward_scores_ragged): img_packed / ev_packed are
        HOST (pinned) [sum len, D] tensors holding only the valid rows of the zero-padded [T, D] chunks, chunk after
        chunk; the chunk / pad rule of data/tools.py:100-114 is applied on the device while ingesting.  valid_lengths:
        host ints [B]; rowmap (int32), chunk_start (int64), chunk_valid (int32): device tensors.  Compact results."""
        import ctypes as C
        lens = [int(v) for v in valid_lengths]
        B, n = len(lens), sum(int(v) for v in valid_lengths)
        if img_packed.is_cuda or ev_packed.is_cuda or img_packed.shape != ev_packed.shape or img_packed.dtype != ev_packed.dtype:
            raise RuntimeError("scores_ragged takes two host tensors of the same shape and dtype")
        if tuple(img_packed.shape) != (n, self.embed_dim) or img_packed.dtype not in _DTYPE_CODES:
            raise RuntimeError(f"packed features must be [{n}, {self.embed_dim}] float32 / float16 / bfloat16")
        if any(v < 0 or v > T for v in lens):
            raise RuntimeError("valid lengths must lie in [0, T]")
        device = _norm_device(device)
        for t, dt, cnt in ((rowmap, torch.int32, n), (chunk_start, torch.int64, B), (chunk_valid, torch.int32, B)):
            if not t.is_cuda or t.dtype != dt or t.numel() != cnt:
                raise RuntimeError("rowmap / chunk_start / chunk_valid must be device tensors (int32 [sum len], int64 [B], int32 [B])")
        img, ev = img_packed.contiguous(), ev_packed.contiguous()
        arr = (C.c_int64 * B)(*lens)
        h, stream = self._prepare(device)
        with torch.cuda.device(device):
            logits = torch.empty(max(n, 1), dtype=torch.float32, device=device)[:n]
            scores = torch.empty(max(n, 1), dtype=torch.float32, device=device)[:n]
            self._set_eval_outputs(h, extra, n, device)
            try:
                _lib.check(_lib.lib.iefvad_model_forward_scores_ragged(
                    h, img.data_ptr(), ev.data_ptr(), _DTYPE_CODES[img.dtype], B, T, C.cast(arr, C.c_void_p), rowmap.data_ptr(),
                    chunk_start.data_ptr(), chunk_valid.data_ptr(), logits.data_ptr(), scores.data_ptr(), stream))
            finally:
                if extra:
                    self._set_eval_outputs(h, None, 0, device)
        return {"logits": logits, "scores": scores, "_keepalive": (img, ev, arr, rowmap, chunk_start, chunk_valid)}

    def scores_from_host(self, img_host: torch.Tensor, ev_host: torch.Tensor, device) -> Dict[str, torch.Tensor]:
        """Host-input evaluation forward on all rows (see `scores`)."""
        if img_host.is_cuda or ev_host.is_cuda:
            raise RuntimeError("scores_from_host takes host tensors; use forward() / scores() for device tensors")
        return self.scores(img_host, ev_host, device)


class MMFMIL(nn.Module):
    """model/imf_vad.py:5-44: holds the bookkeeping attributes and forwards to `self.temporal`."""

    def __init__(self, num_class: int, embed_dim: int, visual_length: int, visual_width: int, visual_head: int,
                 visual_layers: int, attn_window: int, prompt_prefix: int, prompt_postfix: int, device, args):
        super().__init__()
        self.num_class = num_class
        self.visual_length = visual_length
        self.visual_width = visual_width
        self.embed_dim = embed_dim
        self.attn_window = attn_window
        self.prompt_prefix = prompt_prefix
        self.prompt_postfix = prompt_postfix
        self.device = device
        # like the reference (:30-38) the positional visual_head / visual_layers are ignored in favour of args.*
        self.temporal = MultiModal_Fusion_Attn_Iter(
            embed_dim,
            num_layers=args.visual_layers,
            num_heads=args.visual_head,
            num_refinement_steps=args.num_refinement_steps,
            lambda_ref=args.lambda_ref,
            noise_model=args.noise_model,
            nu=args.nu,
        )

    def forward(self, img_visual, ev_visual, padding_mask=None, text=None, lengths=None, return_attn=False):
        # padding_mask / text / lengths / return_attn are accepted and ignored, exactly as at :40-44;
        # the fp16/bf16 -> fp32 cast of :41-42 happens inside the ingest kernel.
        return self.temporal(img_visual, ev_visual)
