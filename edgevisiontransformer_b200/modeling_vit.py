"""Drop-in B200 ViT / DeiT image classifier.

Replaces, for inference, the module the reference evaluates and prunes:
``model(images).logits`` of HF ``ViTForImageClassification`` (deit_pruning/src/utils.py:194-195,
are_16_heads/classifier_eval.py:69-70).  Construct it FROM the (already pruned / optimised) HF module
with :meth:`from_hf`, from an HF-named state dict with :meth:`from_state_dict`, or from a checkpoint
directory with :meth:`from_pretrained` (edgevisiontransformer_b200.checkpoint).  Per-layer head counts and FFN widths
are read off the weight shapes, so nn_pruning / are16heads models with uneven layers load as they are.

The forward runs entirely inside libevt (hand-written sm_100a kernels); torch only owns the tensors.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib


@dataclass
class B200ViTConfig:
    hidden_size: int = 192
    num_hidden_layers: int = 12
    heads: List[int] = field(default_factory=lambda: [3] * 12)          # surviving heads per layer
    intermediate: List[int] = field(default_factory=lambda: [768] * 12)  # FFN width per layer
    head_size: int = 64
    tokens: int = 197
    image_size: int = 224
    patch_size: int = 16
    num_labels: int = 1000
    layer_norm_eps: float = 1e-12
    hidden_act: str = "gelu"          # "gelu" (erf) | "gelu_new"/"gelu_tanh" (tanh)
    dialect: str = "hf"               # "hf" | "tf"
    final_ln: bool = True
    head_hidden: int = 0
    precision: str = "bf16"           # "bf16" (2e-2 logit tolerance) | "tf32" (1e-3; f32 activations)
    embed_k: int = 0                  # >0: caller-built patch matrix with this K (T2T: 576), see forward_embedded
    t2t: int = 0                      # tokens-to-token front-end inside the library (needs embed_k = 576): 1 / True NHWC f32
                                      # pixels (TF T2T), 2 NCHW f32 / bf16 / uint8 pixels (PyTorch T2T, modeling_t2t.B200T2TViTTorch)
    head_rows: int = 1                # 2: DeiTForImageClassificationWithTeacher (cls + distillation rows feed ONE folded classifier)

    # names the reference's callers read off model.config
    @property
    def num_attention_heads(self):
        return max(self.heads)

    @property
    def intermediate_size(self):
        return max(self.intermediate)


@dataclass
class ImageClassifierOutput:
    logits: torch.Tensor
    loss: Optional[torch.Tensor] = None

    def __getitem__(self, i):
        return (self.logits,)[i]


_ACT = {"gelu": _lib.ACT_GELU_ERF, "gelu_erf": _lib.ACT_GELU_ERF, "gelu_new": _lib.ACT_GELU_TANH,
        "gelu_tanh": _lib.ACT_GELU_TANH, "gelu_pytorch_tanh": _lib.ACT_GELU_TANH}
# ("tanh" is deliberately absent: in HF's ACT2FN it names plain nn.Tanh, not the tanh-approximate GELU.)

IMAGENET_DEFAULT_MEAN = (0.485, 0.456, 0.406)   # timm.data.constants, used by deit_pruning/src/utils.py:106-107
IMAGENET_DEFAULT_STD = (0.229, 0.224, 0.225)
_PIX = {torch.float32: _lib.PIX_F32, torch.bfloat16: _lib.PIX_BF16, torch.uint8: _lib.PIX_U8}


def config_from_state_dict(sd: Dict[str, torch.Tensor], *, layer_norm_eps=1e-12, hidden_act="gelu", head_size=64,
                           image_size=224, patch_size=16, dialect="hf", final_ln=None, head_hidden=None,
                           precision="bf16", embed_k=0, t2t=False) -> B200ViTConfig:
    D = sd["vit.embeddings.cls_token"].shape[-1]
    L = 0
    while f"vit.encoder.layer.{L}.attention.attention.query.weight" in sd:
        L += 1
    if L == 0:
        raise ValueError("state dict has no vit.encoder.layer.0.attention.attention.query.weight")
    heads, inter = [], []
    for l in range(L):
        a = sd[f"vit.encoder.layer.{l}.attention.attention.query.weight"].shape[0]
        if a % head_size:
            raise ValueError(f"layer {l}: query rows {a} not a multiple of the head size {head_size}")
        heads.append(a // head_size)
        inter.append(sd[f"vit.encoder.layer.{l}.intermediate.dense.weight"].shape[0])
    if final_ln is None:
        final_ln = "vit.layernorm.weight" in sd
    if head_hidden is None:
        head_hidden = sd["pre_classifier.weight"].shape[0] if "pre_classifier.weight" in sd else 0
    # normalise_keys folds the two heads of a distilled DeiT into one [num_labels, 2 D] classifier over the (cls | distillation) rows
    head_rows = 2 if (not head_hidden and sd["classifier.weight"].shape[-1] == 2 * D) else 1
    return B200ViTConfig(head_rows=head_rows, hidden_size=D, num_hidden_layers=L, heads=heads, intermediate=inter, head_size=head_size,
                         tokens=sd["vit.embeddings.position_embeddings"].shape[-2], image_size=image_size,
                         patch_size=patch_size, num_labels=sd["classifier.weight"].shape[0],
                         layer_norm_eps=layer_norm_eps, hidden_act=hidden_act, dialect=dialect, final_ln=bool(final_ln),
                         head_hidden=int(head_hidden), precision=precision, embed_k=int(embed_k), t2t=int(t2t))


class B200ViTForImageClassification(nn.Module):
    """Inference-only; weights are repacked (bf16, padded) inside libevt at construction."""

    def __init__(self, config: B200ViTConfig, state_dict: Dict[str, torch.Tensor], device=None, max_batch: int = 1024,
                 keep_params: bool = True):
        super().__init__()
        device = torch.device(device if device is not None else "cuda")
        if device.type != "cuda":
            raise RuntimeError("B200ViTForImageClassification runs only on a CUDA (sm_100a) device; no CPU fallback")
        self.config = config
        self.max_batch = int(max_batch)
        self._device = device
        self._lib = _lib.load()
        self._handle = C.c_void_p()
        self._ws: Optional[torch.Tensor] = None
        self._ws_batch = 0
        # Chunks of one call may run on two streams (two workspaces): the persistent GEMMs of the two chunks still take turns on
        # the SMs, but one chunk's LayerNorm (no shared memory, few registers) can sit beside the other chunk's GEMM CTA, and a
        # kernel's tail overlaps the next chunk's kernel instead of idling SMs.  Off unless concurrent_chunks = 2.
        self.concurrent_chunks = int(os.environ.get("EVT_CONCURRENT_CHUNKS", "1"))
        self._ws2: Optional[torch.Tensor] = None
        self._side_stream: Optional[torch.cuda.Stream] = None
        self._graphs: Dict[int, tuple] = {}
        self._ws_listeners: List = []      # called when the workspace is reallocated (dependent CUDA graphs must be dropped)
        self._profiling = False
        # uint8 pixels are normalised inside the patch gather: (x / 255 - mean) / std, the reference loader's transform
        self.pixel_mean: Tuple[float, float, float] = IMAGENET_DEFAULT_MEAN
        self.pixel_std: Tuple[float, float, float] = IMAGENET_DEFAULT_STD
        self._head_mask: Optional[torch.Tensor] = None     # [L, max heads] f32 on the device, set by mask_heads()
        self._capture_ctx = False
        self.context_layers: List[Optional[torch.Tensor]] = []   # per layer [B, heads_l, tokens, 64] after a capturing forward
        spec = _lib.ModelSpec()
        spec.dialect = _lib.DIALECT_TF if config.dialect == "tf" else _lib.DIALECT_HF
        spec.hidden, spec.layers, spec.tokens = config.hidden_size, config.num_hidden_layers, config.tokens
        spec.image, spec.patch, spec.head_size = config.image_size, config.patch_size, config.head_size
        spec.num_labels = config.num_labels
        if config.hidden_act not in _ACT:
            raise ValueError(f"unsupported hidden_act {config.hidden_act!r}")
        spec.act = _ACT[config.hidden_act]
        spec.eps = float(config.layer_norm_eps)
        if config.num_hidden_layers > _lib.MAX_LAYERS:
            raise ValueError("too many layers")
        for l in range(config.num_hidden_layers):
            spec.heads[l] = int(config.heads[l])
            spec.inter[l] = int(config.intermediate[l])
        spec.final_ln = int(config.final_ln)
        spec.head_hidden = int(config.head_hidden)
        spec.t2t = int(config.t2t)
        spec.embed_k = int(config.embed_k)
        spec.head_rows = int(config.head_rows)
        if config.precision not in ("bf16", "tf32"):
            raise ValueError(f"unsupported precision {config.precision!r}")
        spec.precision = _lib.PREC_TF32 if config.precision == "tf32" else _lib.PREC_BF16
        with torch.cuda.device(device):
            _lib.check(self._lib.evt_model_create(C.byref(spec), C.byref(self._handle)), "model_create")
            dev_sd = {k: v.detach().to(device=device, dtype=torch.float32).contiguous() for k, v in state_dict.items()
                      if torch.is_tensor(v) and v.is_floating_point()}
            views = (_lib.TensorView * len(dev_sd))()
            keep = []
            for i, (k, v) in enumerate(dev_sd.items()):
                name = k.encode()
                keep.append(name)
                views[i].name = name
                views[i].data = v.data_ptr()
                views[i].ndim = max(1, min(v.dim(), 4))
                shp = list(v.shape)[-4:] if v.dim() > 4 else list(v.shape)
                if v.dim() > 4:   # collapse leading dims
                    shp[0] = v.numel() // (shp[1] * shp[2] * shp[3])
                for j, s in enumerate(shp or [1]):
                    views[i].shape[j] = s
            _lib.check(self._lib.evt_model_load_weights(self._handle, views, len(dev_sd),
                                                        torch.cuda.current_stream().cuda_stream), "model_load_weights")
        if keep_params:
            self._names = list(dev_sd.keys())
            self._params = nn.ParameterList([nn.Parameter(v, requires_grad=False) for v in dev_sd.values()])
        else:
            self._names = ["classifier.bias"]
            self._params = nn.ParameterList([nn.Parameter(dev_sd["classifier.bias"], requires_grad=False)])
        self.eval()

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_state_dict(cls, sd: Dict[str, torch.Tensor], config: Optional[B200ViTConfig] = None, **kw):
        sd = normalise_keys(sd)
        cfg_kw = {k: kw.pop(k) for k in list(kw) if k in ("layer_norm_eps", "hidden_act", "head_size", "image_size",
                                                            "patch_size", "dialect", "final_ln", "head_hidden", "precision", "embed_k", "t2t")}
        config = config or config_from_state_dict(sd, **cfg_kw)
        return cls(config, sd, **kw)

    @classmethod
    def from_hf(cls, model: nn.Module, **kw):
        """Build from a live HF ViT/DeiT classifier AFTER any surgery (prune_heads, optimize_model):
        shapes come from the module tree (deit_pruning/src/eval_main.py:87-103 order of operations)."""
        hf_cfg = model.config
        sd = normalise_keys({k: v for k, v in model.state_dict().items()})
        config = config_from_state_dict(
            sd, layer_norm_eps=getattr(hf_cfg, "layer_norm_eps", 1e-12), hidden_act=getattr(hf_cfg, "hidden_act", "gelu"),
            head_size=hf_cfg.hidden_size // hf_cfg.num_attention_heads, image_size=_first(hf_cfg.image_size),
            patch_size=_first(hf_cfg.patch_size), precision=kw.pop("precision", "bf16"))
        return cls(config, sd, **kw)

    @classmethod
    def from_timm(cls, model_or_state_dict, **kw):
        """Build from a timm / facebookresearch-deit ``VisionTransformer`` (the model ``utils.get_torch_deit`` returns,
        utils.py:52-62) or its state dict: fused qkv, LayerNorm eps 1e-6 (dialects.timm_vit_to_canonical).  DeiT III
        (``models_v2`` / timm ``deit3_*``, LayerScale) loads too.  The patch size is read from the patch projection; the head
        size (not in the weights) defaults to 64, or to 80 for a DeiT III of embed dim 1280 (Huge); ``head_size=`` overrides."""
        from .dialects import deit3_head_size, timm_vit_to_canonical
        sd = model_or_state_dict.state_dict() if hasattr(model_or_state_dict, "state_dict") else model_or_state_dict
        sd = {k: v for k, v in sd.items()}
        image = kw.pop("image_size", None)
        head_size = kw.pop("head_size", None)
        inner = sd["model"] if isinstance(sd.get("model"), dict) else sd
        patch = kw.pop("patch_size", None)
        if patch is None:
            patch = inner["patch_embed.proj.weight"].shape[-1] if "patch_embed.proj.weight" in inner else 16
        csd, cfg_kw = timm_vit_to_canonical(sd, patch=patch)
        cfg_kw["head_size"] = deit3_head_size(sd) if head_size is None else int(head_size)
        if image is None:                       # from the position rows: 197 / 198 -> 224, 577 / 578 -> 384
            n_prefix = 2 if "vit.embeddings.distillation_token" in csd else 1
            image = int(round((csd["vit.embeddings.position_embeddings"].shape[1] - n_prefix) ** 0.5)) * cfg_kw["patch_size"]
        return cls.from_state_dict(csd, image_size=image, **cfg_kw, **kw)

    @classmethod
    def from_pretrained(cls, model_dir: str, **kw):
        from .checkpoint import load_checkpoint
        sd, cfg_kw = load_checkpoint(model_dir)
        cfg_kw.update({k: kw.pop(k) for k in list(kw) if k in ("hidden_act", "layer_norm_eps", "precision")})
        return cls.from_state_dict(sd, **cfg_kw, **kw)

    # ------------------------------------------------------------------ nn.Module surface
    def num_parameters(self, only_trainable: bool = False) -> int:
        return 0 if only_trainable else sum(p.numel() for p in self._params)

    def state_dict(self, *a, **kw):  # HF-named view of the weights this model was built from
        return {n: p.detach() for n, p in zip(self._names, self._params)}

    def to(self, *args, **kwargs):
        dev = None
        for a in args:
            if isinstance(a, (str, torch.device)):
                dev = torch.device(a)
        dev = torch.device(kwargs["device"]) if "device" in kwargs else dev
        if dev is not None and (dev.type != "cuda" or (dev.index is not None and dev.index != self._device.index
                                                       and self._device.index is not None)):
            raise RuntimeError("B200ViTForImageClassification is bound to its CUDA device; rebuild it to move it")
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda" if device is None else device))

    def train(self, mode: bool = True):
        if mode:
            raise RuntimeError("B200ViTForImageClassification is inference-only")
        return super().train(False)

    def __del__(self):
        try:
            if getattr(self, "_handle", None) is not None and self._handle.value:
                self._lib.evt_model_destroy(self._handle)
                self._handle = C.c_void_p()
        except Exception:
            pass

    # ------------------------------------------------------------------ forward
    def _workspace(self, batch: int) -> torch.Tensor:
        if self._ws is None or batch > self._ws_batch:
            n = C.c_size_t()
            _lib.check(self._lib.evt_model_workspace_bytes(self._handle, batch, C.byref(n)), "workspace_bytes")
            self._ws = torch.empty(n.value, dtype=torch.uint8, device=self._device)
            self._ws_batch = batch
            self._graphs.clear()
            for cb in self._ws_listeners:    # graphs captured by wrappers (T2T front-end) hold the old workspace pointer
                cb()
        return self._ws

    def on_workspace_realloc(self, callback) -> None:
        """Register a callable invoked whenever the activation workspace is reallocated: anything that baked the old
        pointer into a CUDA graph (modeling_t2t.B200T2TViT.forward_graphed) must drop it."""
        self._ws_listeners.append(callback)

    def _run(self, pixels: torch.Tensor, logits: torch.Tensor, ws: Optional[torch.Tensor] = None,
             head_mask: Optional[torch.Tensor] = None, ctx: Optional[List[torch.Tensor]] = None) -> None:
        B = pixels.shape[0]
        if ws is None:
            ws = self._workspace(B)
        stream = torch.cuda.current_stream().cuda_stream
        if pixels.dtype == torch.float32 and head_mask is None and ctx is None:
            _lib.check(self._lib.evt_model_forward(self._handle, pixels.data_ptr(), B, logits.data_ptr(), ws.data_ptr(),
                                                   ws.numel(), stream), "model_forward")
            return
        opts = _lib.ForwardOpts()
        opts.pixel_dtype = _PIX[pixels.dtype]
        for c in range(3):
            opts.pixel_scale[c] = 1.0 / (255.0 * self.pixel_std[c])
            opts.pixel_bias[c] = -self.pixel_mean[c] / self.pixel_std[c]
        if head_mask is not None:
            opts.head_mask = head_mask.data_ptr()
            opts.head_mask_ld = head_mask.stride(0)
        if ctx is not None:
            arr = (C.c_void_p * len(ctx))(*[t.data_ptr() for t in ctx])
            opts.ctx_out = C.cast(arr, C.POINTER(C.c_void_p))
        _lib.check(self._lib.evt_model_forward_ex(self._handle, pixels.data_ptr(), C.byref(opts), B, logits.data_ptr(),
                                                  ws.data_ptr(), ws.numel(), stream), "model_forward_ex")

    # ------------------------------------------------------------------ are_16_heads surface
    @property
    def vit(self):
        """`model.vit.mask_heads(to_prune)` is how are_16_heads/run_classifier.py:247-250 reaches the encoder."""
        return self

    def mask_heads(self, heads_to_mask: Optional[Dict[int, object]]) -> None:
        """Zero the context of the given heads, {layer: iterable of head indices}, in every later forward (the heads stay
        in the weights: are_16_heads' masking-instead-of-pruning mode).  None or {} clears the mask."""
        if not heads_to_mask:
            self._head_mask = None
            return
        c = self.config
        m = torch.ones((c.num_hidden_layers, max(c.heads)), dtype=torch.float32)
        for layer, hs in heads_to_mask.items():
            for h in hs:
                if not (0 <= int(layer) < c.num_hidden_layers and 0 <= int(h) < c.heads[int(layer)]):
                    raise ValueError(f"mask_heads: head {h} of layer {layer} does not exist")
                m[int(layer), int(h)] = 0.0
        self._head_mask = m.to(self._device)

    def capture_context(self, enable: bool = True) -> None:
        """Keep every layer's attention context of the next forwards in `context_layers[l]` ([B, heads_l, tokens, 64],
        the `context_layer_val` that are_16_heads/classifier_eval.py:183-191 reads for the head-importance score)."""
        self._capture_ctx = bool(enable)
        if not enable:
            self.context_layers = []

    def _resolve_head_mask(self, head_mask) -> Optional[torch.Tensor]:
        """HF semantics (get_head_mask): [heads] applies to every layer, [layers, heads] per layer; multiplied into the
        attention probabilities of a head, i.e. into its context.  Combined with mask_heads()."""
        c = self.config
        hm = self._head_mask
        if head_mask is not None:
            m = torch.as_tensor(head_mask, dtype=torch.float32, device=self._device)
            if m.dim() == 1:
                m = m.unsqueeze(0).expand(c.num_hidden_layers, -1)
            if m.dim() != 2 or m.shape[0] != c.num_hidden_layers or m.shape[1] < max(c.heads):
                raise ValueError(f"head_mask must be [heads] or [layers, heads] with heads >= {max(c.heads)}")
            m = m[:, :max(c.heads)]
            hm = m if hm is None else hm * m
        return hm.contiguous() if hm is not None else None

    def _run_chunks_two_streams(self, x: torch.Tensor, logits: torch.Tensor) -> None:
        """Even chunks on the current stream, odd chunks on a side stream with a second workspace."""
        B = x.shape[0]
        ws = self._workspace(self.max_batch)
        if self._ws2 is None or self._ws2.numel() < ws.numel():
            self._ws2 = torch.empty_like(ws)
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self._device)
        main, side = torch.cuda.current_stream(), self._side_stream
        side.wait_stream(main)                       # inputs / output buffer are ready on the side stream too
        for i, s in enumerate(range(0, B, self.max_batch)):
            e = min(B, s + self.max_batch)
            if i & 1:
                with torch.cuda.stream(side):
                    self._run(x[s:e], logits[s:e], self._ws2)
            else:
                self._run(x[s:e], logits[s:e], ws)
        main.wait_stream(side)

    @torch.no_grad()
    def forward(self, pixel_values: Optional[torch.Tensor] = None, head_mask=None, labels=None, output_attentions=None,
                output_hidden_states=None, interpolate_pos_encoding=None, return_dict=None) -> ImageClassifierOutput:
        """HF `ViTForImageClassification.forward` surface (SITE/models/vit/modeling_vit.py:620-653).  pixel_values may be
        f32, bf16 or uint8 (uint8 is normalised with pixel_mean / pixel_std inside the patch gather).  Options this
        inference path does not implement raise instead of being ignored."""
        if pixel_values is None:
            raise ValueError("You have to specify pixel_values")
        for name, v in (("labels", labels), ("output_attentions", output_attentions),
                        ("output_hidden_states", output_hidden_states), ("interpolate_pos_encoding", interpolate_pos_encoding)):
            if v is not None and v is not False:
                raise NotImplementedError(f"B200ViTForImageClassification.forward does not support {name}")
        x = pixel_values
        if not x.is_cuda:
            raise RuntimeError("pixel_values must be a CUDA tensor (no CPU fallback); move the batch with .to(device)")
        c = self.config
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != c.image_size or x.shape[3] != c.image_size:
            raise ValueError(f"Input image size ({tuple(x.shape[2:])}) doesn't match model ({c.image_size}*{c.image_size}).")
        if x.dtype not in _PIX:
            x = x.float()
        x = x.contiguous()
        B = x.shape[0]
        logits = torch.empty((B, c.num_labels), dtype=torch.float32, device=x.device)
        hm = self._resolve_head_mask(head_mask)
        ctx_all = None
        if self._capture_ctx:
            cdt = torch.float32 if c.precision == "tf32" else torch.bfloat16
            ctx_all = [torch.empty((B * c.tokens, h * c.head_size), dtype=cdt, device=x.device) for h in c.heads]
        with torch.cuda.device(self._device):
            if self.concurrent_chunks >= 2 and B > self.max_batch and not self._profiling and hm is None and ctx_all is None:
                self._run_chunks_two_streams(x, logits)
            else:
                for s in range(0, B, self.max_batch):
                    e = min(B, s + self.max_batch)
                    ctx = [t[s * c.tokens:e * c.tokens] for t in ctx_all] if ctx_all is not None else None
                    self._run(x[s:e], logits[s:e], head_mask=hm, ctx=ctx)
        if ctx_all is not None:
            self.context_layers = [t.view(B, c.tokens, h, c.head_size).permute(0, 2, 1, 3) for t, h in zip(ctx_all, c.heads)]
        return ImageClassifierOutput(logits=logits)

    @torch.no_grad()
    def forward_embedded(self, patch_matrix: torch.Tensor) -> ImageClassifierOutput:
        """Forward from the A operand of the token-embedding GEMM ([B*patches, ld], operand dtype): the entry the T2T
        front-end uses (its last soft split IS that matrix)."""
        c = self.config
        patches = c.tokens - 1 if c.tokens == (c.image_size // c.patch_size) ** 2 + 1 else c.tokens - 2
        if not patch_matrix.is_cuda or patch_matrix.dim() != 2 or patch_matrix.stride(1) != 1 or patch_matrix.shape[0] % patches:
            raise ValueError("forward_embedded wants a CUDA [B*patches, ld] matrix")
        want = torch.float32 if c.precision == "tf32" else torch.bfloat16
        if patch_matrix.dtype != want:
            raise ValueError(f"forward_embedded wants {want} for precision {c.precision}")
        B = patch_matrix.shape[0] // patches
        logits = torch.empty((B, c.num_labels), dtype=torch.float32, device=patch_matrix.device)
        with torch.cuda.device(self._device):
            for s in range(0, B, self.max_batch):
                e = min(B, s + self.max_batch)
                ws = self._workspace(e - s)
                pm = patch_matrix[s * patches:e * patches]
                _lib.check(self._lib.evt_model_forward_embedded(self._handle, pm.data_ptr(), pm.stride(0), e - s,
                                                                logits[s:e].data_ptr(), ws.data_ptr(), ws.numel(),
                                                                torch.cuda.current_stream().cuda_stream), "model_forward_embedded")
        return ImageClassifierOutput(logits=logits)

    # ------------------------------------------------------------------ latency path: CUDA graph
    @torch.no_grad()
    def forward_graphed(self, pixel_values: torch.Tensor) -> ImageClassifierOutput:
        """Same result as forward(); the launch sequence for this batch size is captured once in a CUDA graph
        and replayed, removing per-kernel launch overhead at small batch."""
        B = pixel_values.shape[0]
        if B > self.max_batch or self._head_mask is not None or self._capture_ctx:
            return self.forward(pixel_values)
        ent = self._graphs.get(B)
        with torch.cuda.device(self._device):
            if ent is None:
                self._workspace(B)
                static_in = torch.empty((B, 3, self.config.image_size, self.config.image_size), dtype=torch.float32,
                                        device=self._device)
                static_out = torch.empty((B, self.config.num_labels), dtype=torch.float32, device=self._device)
                static_in.copy_(pixel_values)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(2):
                        self._run(static_in, static_out)
                torch.cuda.current_stream().wait_stream(side)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._run(static_in, static_out)
                ent = (g, static_in, static_out)
                self._graphs[B] = ent
            g, static_in, static_out = ent
            static_in.copy_(pixel_values)
            g.replay()
            return ImageClassifierOutput(logits=static_out.clone())

    def launches_per_forward(self) -> int:
        return int(self._lib.evt_model_launches_per_forward(self._handle))

    # ------------------------------------------------------------------ measurement aid
    def profile_begin(self) -> None:
        """Forwards issued from now on record a CUDA event after every launch (evt_model_profile_begin)."""
        _lib.check(self._lib.evt_model_profile_begin(self._handle), "profile_begin")
        self._profiling = True

    def profile_end(self) -> Dict[str, Tuple[float, int]]:
        """-> {stage: (summed device ms, launches)} over the forwards since profile_begin(); synchronises."""
        n = len(_lib.STAGES)
        ms, cnt = (C.c_float * n)(), (C.c_int * n)()
        self._profiling = False
        _lib.check(self._lib.evt_model_profile_end(self._handle, ms, cnt), "profile_end")
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(_lib.STAGES)}


# DeiT III (facebookresearch-deit models_v2 ``deit_*_LS``, timm ``deit3_*``): name -> (embed dim, heads, patch, image size).
# Depth comes from the weights.
DEIT3 = {
    "deit3_small_patch16_224": (384, 6, 16, 224), "deit3_small_patch16_384": (384, 6, 16, 384),
    "deit3_medium_patch16_224": (512, 8, 16, 224), "deit3_medium_patch16_384": (512, 8, 16, 384),
    "deit3_base_patch16_224": (768, 12, 16, 224), "deit3_base_patch16_384": (768, 12, 16, 384),
    "deit3_large_patch16_224": (1024, 16, 16, 224), "deit3_large_patch16_384": (1024, 16, 16, 384),
    "deit3_huge_patch14_224": (1280, 16, 14, 224),
}


def _deit3_factory(name: str, checkpoint_or_sd, **kw) -> B200ViTForImageClassification:
    """A DeiT III checkpoint (file or state dict, either key layout) as the named model: its shapes must match the name."""
    from .dialects import _LAYERSCALE, _refuse_deit3_variants, unwrap_checkpoint
    D, heads, patch, image = DEIT3[name]
    sd = checkpoint_or_sd
    if isinstance(sd, (str, os.PathLike)):
        sd = torch.load(sd, map_location="cpu", weights_only=True)
    sd = unwrap_checkpoint(sd)
    _refuse_deit3_variants(sd)
    if not any(_LAYERSCALE.search(k) for k in sd):
        raise ValueError(f"{name} is a DeiT III (LayerScale) model; the weights have no blocks.*.gamma_1 / ls1.gamma")
    got = (sd["cls_token"].shape[-1], sd["patch_embed.proj.weight"].shape[-1], sd["blocks.0.mlp.fc1.weight"].shape[0])
    if got != (D, patch, 4 * D):
        raise ValueError(f"{name} is embed dim {D}, patch {patch}, MLP {4 * D}; the weights have {got[0]}, {got[1]} and {got[2]}")
    n, patches = sd["pos_embed"].shape[-2], (image // patch) ** 2
    if n not in (patches, patches + 1):
        raise ValueError(f"{name} has {patches} patches; the weights have {n} position rows")
    kw.setdefault("image_size", image)
    return B200ViTForImageClassification.from_timm(sd, patch_size=patch, head_size=D // heads, **kw)


def deit3_small_patch16_224(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_small_patch16_224", checkpoint_or_sd, **kw)


def deit3_small_patch16_384(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_small_patch16_384", checkpoint_or_sd, **kw)


def deit3_medium_patch16_224(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_medium_patch16_224", checkpoint_or_sd, **kw)


def deit3_medium_patch16_384(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_medium_patch16_384", checkpoint_or_sd, **kw)


def deit3_base_patch16_224(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_base_patch16_224", checkpoint_or_sd, **kw)


def deit3_base_patch16_384(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_base_patch16_384", checkpoint_or_sd, **kw)


def deit3_large_patch16_224(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_large_patch16_224", checkpoint_or_sd, **kw)


def deit3_large_patch16_384(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_large_patch16_384", checkpoint_or_sd, **kw)


def deit3_huge_patch14_224(checkpoint_or_sd, **kw):
    return _deit3_factory("deit3_huge_patch14_224", checkpoint_or_sd, **kw)


def _first(v):
    return v[0] if isinstance(v, (tuple, list)) else v


def normalise_keys(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Accept HF ViT ('vit.'), HF DeiT ('deit.') and DDP ('module.') prefixes.

    HF `DeiTForImageClassification` (198 tokens: cls + distillation token, ONE classifier on the cls row,
    SITE/models/deit/modeling_deit.py:595-659) loads as it is.  `DeiTForImageClassificationWithTeacher` (the layout of the
    public `facebook/deit-*-distilled-*` checkpoints) answers with the MEAN of `cls_classifier(cls row)` and
    `distillation_classifier(distillation row)`: its two heads are folded here into one classifier over the concatenated
    (cls | distillation) rows, `classifier.weight = [W_cls | W_dist] / 2`, `classifier.bias = (b_cls + b_dist) / 2`, which the
    runtime evaluates as a single GEMM with K = 2 D (`evt_model_spec.head_rows = 2`).  Half of such a pair is refused."""
    out = {}
    for k, v in sd.items():
        if k.startswith("module."):
            k = k[len("module."):]
        if k.startswith("deit."):
            k = "vit." + k[len("deit."):]
        out[k] = v
    two = [k for k in out if k.startswith(("cls_classifier.", "distillation_classifier."))]
    if two:
        need = {"cls_classifier.weight", "cls_classifier.bias", "distillation_classifier.weight", "distillation_classifier.bias"}
        if set(two) != need or "classifier.weight" in out:
            raise ValueError("distilled DeiT checkpoint (DeiTForImageClassificationWithTeacher) needs cls_classifier and "
                             f"distillation_classifier weight + bias and no third head; found {sorted(two)}")
        wc, wd = out.pop("cls_classifier.weight"), out.pop("distillation_classifier.weight")
        bc, bd = out.pop("cls_classifier.bias"), out.pop("distillation_classifier.bias")
        if wc.shape != wd.shape:
            raise ValueError("distilled DeiT checkpoint: the two heads differ in shape")
        out["classifier.weight"] = torch.cat((wc.float(), wd.float()), dim=1) * 0.5
        out["classifier.bias"] = (bc.float() + bd.float()) * 0.5
    return out
