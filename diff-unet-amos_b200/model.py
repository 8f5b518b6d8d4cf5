"""Drop-in ``DiffUNet`` for the reference's inference path, backed by libdunet_b200.so.

Mirrors the Python seams of the reference (SURVEY.md 8b):

  * ``DiffUNetB200(spatial_dims, in_channels, out_channels, image_size, spatial_size, features, dropout, timesteps,
    mode)``                                  -> models/diff_unet.py:10-21
  * ``forward(image=, x=, step=, pred_type=)`` with pred_type in {"q_sample", "denoise", "ddim_sample"}, anything else
    raises NotImplementedError             -> models/diffusion/diffusion.py:49-63
  * attributes ``embed_model``, ``model``, ``diffusion``, ``sample_diffusion``, ``sampler``, ``num_classes``
                                             -> models/diffusion/diffusion.py:25-47
  * ``model(x, t, image=, embeddings=)``     -> models/basic_unet/denoiser.py:284-312
  * ``embed_model(image)`` -> 5 feature maps -> models/basic_unet/pretrained/basic_unet.py:496-512
  * ``sample_diffusion.ddim_sample_loop(model, shape, noise=, model_kwargs=)`` -> gaussian_diffusion.py:626-665
  * ``state_dict`` / ``load_state_dict`` with the reference's checkpoint keys (SURVEY Appendix F)

All tensor math runs in the CUDA library; this file only owns parameters, buffers and call sequencing.  There is no
CPU path: calling a compute method with CPU tensors raises.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .schedule import DdimSchedule

DEFAULT_FEATURES = (64, 64, 128, 256, 512, 64)
PRECISIONS = ("fp16", "bf16", "fp32x3")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the B200 path has no CPU fallback")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class _Node(nn.Module):
    """Bare container so parameters get the reference's dotted checkpoint names."""


def _attach(root: nn.Module, dotted: str, tensor: torch.Tensor) -> None:
    *path, leaf = dotted.split(".")
    node = root
    for part in path:
        if part not in node._modules:
            node.add_module(part, _Node())
        node = node._modules[part]
    node.register_parameter(leaf, nn.Parameter(tensor, requires_grad=False))


def _init_like_reference(root: nn.Module, in_channels: int, out_channels: int, f: Sequence[int]) -> None:
    """Create parameters with PyTorch's default initialisers in the reference's construction order, so that
    ``torch.manual_seed(s); DiffUNetB200(...)`` holds the same values as ``torch.manual_seed(s); DiffUNet(...)``."""

    def conv(prefix, cin, cout, k):
        m = nn.Conv3d(cin, cout, k, padding=k // 2)
        _attach(root, prefix + ".weight", m.weight.detach())
        _attach(root, prefix + ".bias", m.bias.detach())

    def block(prefix, cin, cout):
        conv(prefix + ".conv", cin, cout, 3)
        _attach(root, prefix + ".adn.N.weight", torch.ones(cout))
        _attach(root, prefix + ".adn.N.bias", torch.zeros(cout))

    def linear(prefix, cin, cout):
        m = nn.Linear(cin, cout)
        _attach(root, prefix + ".weight", m.weight.detach())
        _attach(root, prefix + ".bias", m.bias.detach())

    def twoconv(prefix, cin, cout, temb):
        if temb:
            linear(prefix + ".temb_proj", 512, cout)
        block(prefix + ".conv_0", cin, cout)
        block(prefix + ".conv_1", cout, cout)

    twoconv("embed_model.conv_0", in_channels, f[0], False)
    for d in range(4):
        twoconv(f"embed_model.down.{d}.convs", f[d], f[d + 1], False)
    linear("model.temb.dense.0", 128, 512)
    linear("model.temb.dense.1", 512, 512)
    twoconv("model.conv_0", in_channels + out_channels, f[0], True)
    for lvl in range(1, 5):
        twoconv(f"model.down_{lvl}.convs", f[lvl - 1], f[lvl], True)
    for lvl, cin, ccat, cout, halves in ((4, f[4], f[3], f[3], True), (3, f[3], f[2], f[2], True),
                                         (2, f[2], f[1], f[1], True), (1, f[1], f[0], f[5], False)):
        cup = cin // 2 if halves else cin
        m = nn.ConvTranspose3d(cin, cup, 2, stride=2)
        _attach(root, f"model.upcat_{lvl}.upsample.deconv.weight", m.weight.detach())
        _attach(root, f"model.upcat_{lvl}.upsample.deconv.bias", m.bias.detach())
        twoconv(f"model.upcat_{lvl}.convs", ccat + cup, cout, True)
    conv("model.final_conv", f[5], out_channels, 1)


class _UniformSampler:
    """``UniformSampler(timesteps)`` (guided_diffusion/resample.py:61-66 + ScheduleSampler.sample): training only."""

    def __init__(self, n):
        self.n = n

    def sample(self, batch_size, device):
        idx = torch.randint(0, self.n, (batch_size,), device=device)
        return idx, torch.ones(batch_size, device=device)


class _TrainDiffusion:
    """The 1000-step process used by ``q_sample`` (models/diffusion/diffusion.py:31-36,65-69): fp32-cast tables of the
    linear schedule on the device + the CUDA ``q_sample`` kernel (gaussian_diffusion.py:187-205)."""

    def __init__(self, timesteps):
        betas = np.linspace(1000 / timesteps * 1e-4, 1000 / timesteps * 0.02, timesteps, dtype=np.float64)
        ac = np.cumprod(1.0 - betas)
        self.num_timesteps = timesteps
        self.sqrt_alphas_cumprod = np.sqrt(ac)
        self.sqrt_one_minus_alphas_cumprod = np.sqrt(1.0 - ac)
        self._dev = {}

    def _tables(self, device):
        if device not in self._dev:
            self._dev[device] = (torch.from_numpy(self.sqrt_alphas_cumprod).float().to(device),
                                 torch.from_numpy(self.sqrt_one_minus_alphas_cumprod).float().to(device))
        return self._dev[device]

    def q_sample(self, x_start, t, noise=None, seed: int = 0, stream_id: int = 0, return_noise: bool = False):
        x_start = _f32c(x_start, "x_start")
        t = t.to(device=x_start.device, dtype=torch.int64).contiguous()
        if int(t.min()) < 0 or int(t.max()) >= self.num_timesteps:
            raise IndexError(f"timesteps must lie in [0, {self.num_timesteps})")
        a, b = self._tables(x_start.device)
        out = torch.empty_like(x_start)
        nz_out = None
        if noise is None:
            nz_out = torch.empty_like(x_start)
        else:
            noise = _f32c(noise, "noise")
            assert noise.shape == x_start.shape
        B = x_start.shape[0]
        with torch.cuda.device(x_start.device):
            _lib.check(_lib.load().dunet_q_sample(_ptr(x_start), _ptr(noise), _ptr(nz_out), _ptr(t), _ptr(a), _ptr(b), _ptr(out), B,
                                                  x_start[0].numel(), ctypes.c_uint64(seed & (2 ** 64 - 1)), int(stream_id), _stream()))
        if return_noise:
            return out, (noise if noise is not None else nz_out)
        return out


class _Runtime:
    """Owns the dunet_plan, the packed-weight freshness check and the per-batch workspaces of one DiffUNetB200."""

    def __init__(self, owner: "DiffUNetB200"):
        self.owner = owner
        self.plan = None
        self.device = None
        self.weights_sig = None
        self.workspaces: Dict[str, torch.Tensor] = {}
        self.ws_batch = None   # batch size of the last call that used the workspace
        self.emb_token = None  # identity of the embeddings currently held in the workspace

    def close(self):
        if self.plan is not None:
            _lib.load().dunet_plan_destroy(self.plan)
            self.plan = None

    def _signature(self):
        return tuple((p.data_ptr(), p._version) for p in self.owner.parameters())

    def ensure(self, device: torch.device):
        o = self.owner
        lib = _lib.load()
        if self.plan is None or self.device != device:
            self.close()
            cfg = _lib.DunetCfg()
            cfg.num_classes, cfg.in_channels = o.num_classes, o.in_channels
            cfg.patch = (ctypes.c_int32 * 3)(*o.patch)
            cfg.features = (ctypes.c_int32 * 6)(*o.features)
            cfg.batch_max, cfg.num_steps, cfg.flags = o.batch_max, o.num_steps, o.debug_flags
            plan = ctypes.c_void_p()
            with torch.cuda.device(device):
                _lib.check(lib.dunet_plan_create(ctypes.byref(plan), ctypes.byref(cfg)))
            self.plan, self.device, self.weights_sig = plan, device, None
            self.workspaces.clear()
            s = o.schedule
            n = s.num_timesteps
            _lib.check(lib.dunet_plan_set_schedule(
                plan, n, (ctypes.c_int32 * n)(*s.timestep_map),
                (ctypes.c_float * n)(*s.sqrt_recip_alphas_cumprod.astype(np.float32)),
                (ctypes.c_float * n)(*s.sqrt_recipm1_alphas_cumprod.astype(np.float32)),
                (ctypes.c_float * n)(*s.alphas_cumprod_prev.astype(np.float32))))
        sig = self._signature()
        if sig != self.weights_sig:
            with torch.cuda.device(device):
                for key, p in o.state_dict().items():
                    if p.device != device or p.dtype != torch.float32:
                        raise RuntimeError(f"parameter {key} must be fp32 on {device}; move the module with .to(device)")
                    t = p.contiguous()
                    shape = (ctypes.c_int64 * t.dim())(*t.shape)
                    _lib.check(lib.dunet_plan_set_weight(self.plan, key.encode(), _ptr(t), shape, t.dim(), _stream()))
                _lib.check(lib.dunet_plan_commit(self.plan, _stream()))
            self.weights_sig = sig
            self.emb_token = None
        return self.plan

    def workspace(self, batch: int) -> torch.Tensor:
        """ONE workspace, sized for the largest batch (any smaller batch lays itself out inside it), so alternating batch
        sizes (the last, shorter window group of every volume) never re-allocate.  The embeddings it holds are tied to
        the batch size they were written with: a change of batch size invalidates them."""
        ws = self.workspaces.get("max")
        if ws is None:
            lib = _lib.load()
            need = 0
            for b in range(1, self.owner.batch_max + 1):
                nbytes = ctypes.c_size_t()
                _lib.check(lib.dunet_workspace_bytes(self.plan, b, ctypes.byref(nbytes)))
                need = max(need, nbytes.value)
            buf = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
            off = (-buf.data_ptr()) % 256
            ws = buf[off:off + need]
            self.workspaces["max"] = ws
            self.ws_batch = None
        if self.ws_batch != batch:
            self.ws_batch = batch
            self.emb_token = None
        return ws


class EncoderB200(nn.Module):
    """``BasicUNetEncoder`` seam: forward(image) -> [x0..x4] fp32 NCDHW."""

    def __init__(self, owner):
        super().__init__()
        object.__setattr__(self, "_owner", owner)

    def forward(self, x: torch.Tensor) -> List[torch.Tensor]:
        o = self._owner
        image = _f32c(x, "image")
        o._check_image(image)
        rt = o._rt
        plan = rt.ensure(image.device)
        B = image.shape[0]
        ws = rt.workspace(B)
        lib = _lib.load()
        with torch.cuda.device(image.device):
            _lib.check(lib.dunet_encode(plan, _ptr(image), B, _ptr(ws), _stream()))
            outs = []
            for lvl in range(5):
                shp = (B, o.features[lvl]) + tuple(s >> lvl for s in o.patch)
                t = torch.empty(shp, dtype=torch.float32, device=image.device)
                _lib.check(lib.dunet_get_embedding(plan, lvl, _ptr(t), B, _ptr(ws), _stream()))
                outs.append(t)
        rt.emb_token = (tuple(id(t) for t in outs), B)
        o._emb_keepalive = outs
        return outs


class DenoiserB200(nn.Module):
    """``BasicUNetRDenoiser`` seam: forward(x, t, image=, embeddings=) -> logits fp32 NCDHW."""

    def __init__(self, owner):
        super().__init__()
        object.__setattr__(self, "_owner", owner)

    def parameters(self, recurse: bool = True):  # ddim_sample_loop takes next(model.parameters()).device
        return self._owner._modules["model_params"].parameters(recurse)

    def forward(self, x: torch.Tensor, t: torch.Tensor, image: torch.Tensor = None, embeddings=None) -> torch.Tensor:
        o = self._owner
        if image is None or embeddings is None:
            raise ValueError("model(x, t, image=, embeddings=) needs both image and embeddings (denoiser.py:298-304)")
        x = _f32c(x, "x")
        image = _f32c(image, "image")
        o._check_image(image)
        B = x.shape[0]
        tv = [int(v) for v in torch.as_tensor(t).reshape(-1).tolist()]
        if len(tv) == 1:
            tv = tv * B
        if len(tv) != B:
            raise ValueError(f"t must hold one timestep per sample ({B}), got {len(tv)}")
        rt = o._rt
        plan = rt.ensure(x.device)
        ws = rt.workspace(B)
        o._upload_embeddings(embeddings, B, ws)
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().dunet_denoise_step(plan, _ptr(x), _ptr(image), (ctypes.c_int32 * B)(*tv), _ptr(out), B, _ptr(ws),
                                                      _stream()))
        return out


class SmoothUNetDenoiserB200(DenoiserB200):
    """``SmoothUNetDenoiser`` seam (models/smooth_unet/denoiser.py:9-61, SURVEY 8f-2).  Its ``forward`` (:41-61) is the same
    graph as ``BasicUNetRDenoiser.forward`` -- time embedding, cat([image, x]), five TwoConv levels + encoder residuals, four
    UpCat blocks, final 1x1x1 conv -- so it runs on the same kernels; this class only mirrors the keyword order of the
    reference signature ``forward(x, t, embeddings=None, image=None)``.

    ``norm``: the reference class defaults to ``("layer", {"affine": True})`` (:17).  MONAI's ``get_norm_layer`` turns that
    into ``nn.LayerNorm(affine=True)`` -- LayerNorm has neither a ``num_features`` nor an ``affine`` argument and needs a
    ``normalized_shape`` the factory never supplies -- so the default cannot be constructed (TypeError) and no reference
    behaviour exists to match.  Only ``norm="instance"`` (what BasicUNetRDenoiser uses, denoiser.py:206-209) is accepted."""

    def __init__(self, owner, norm="instance", smoothing: bool = False):
        name = norm[0] if isinstance(norm, (tuple, list)) else norm
        if str(name).lower() != "instance":
            raise NotImplementedError(
                f"norm={norm!r}: the reference's default ('layer') is not constructible through MONAI's norm factory "
                "(nn.LayerNorm(affine=True) raises); only the instance-norm graph is defined")
        super().__init__(owner)
        self.smoothing = smoothing

    def forward(self, x: torch.Tensor, t: torch.Tensor, embeddings=None, image: torch.Tensor = None) -> torch.Tensor:
        return super().forward(x, t, image=image, embeddings=embeddings)


class SampleDiffusionB200:
    """``SpacedDiffusion`` seam for sampling: tables + ``ddim_sample_loop`` (gaussian_diffusion.py:626-665)."""

    def __init__(self, owner):
        self._owner = owner
        s = owner.schedule
        self.timestep_map = list(s.timestep_map)
        self.num_timesteps = s.num_timesteps
        self.alphas_cumprod = s.alphas_cumprod
        self.alphas_cumprod_prev = s.alphas_cumprod_prev
        self.sqrt_recip_alphas_cumprod = s.sqrt_recip_alphas_cumprod
        self.sqrt_recipm1_alphas_cumprod = s.sqrt_recipm1_alphas_cumprod

    def ddim_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                         model_kwargs=None, device=None, progress=False, eta=0.0):
        o = self._owner
        if model is not o.model:
            raise NotImplementedError("the fused sampler only drives this module's own denoiser")
        if not clip_denoised or denoised_fn is not None or cond_fn is not None or eta != 0.0:
            raise NotImplementedError("only the branch the reference takes is implemented: clip_denoised, eta = 0")
        kw = model_kwargs or {}
        image, embeddings = kw.get("image"), kw.get("embeddings")
        if image is None or embeddings is None:
            raise ValueError("model_kwargs must carry image and embeddings (models/diffusion/diffusion.py:91-93)")
        image = _f32c(image, "image")
        if noise is None:
            noise = torch.randn(*shape, device=image.device)  # gaussian_diffusion.py:693
        noise = _f32c(noise, "noise")
        B = noise.shape[0]
        rt = o._rt
        plan = rt.ensure(image.device)
        ws = rt.workspace(B)
        o._upload_embeddings(embeddings, B, ws)
        res = o._run_ddim(image, noise, run_encoder=False, want_steps=True)
        outs = res["per_step"]
        n = self.num_timesteps
        all_out = [outs[k].cpu() for k in range(n)]            # reference moves every step to the host (:660-661)
        all_x0 = [t.clamp(-1, 1) for t in all_out]
        return {"sample": res["final_x"], "pred_xstart": outs[n - 1].clamp(-1, 1), "model_output": outs[n - 1],
                "all_samples": all_x0, "all_model_outputs": all_out}


class DiffUNetB200(nn.Module):
    def __init__(self, spatial_dims: int = 3, in_channels: int = 3, out_channels: int = 1, image_size=96,
                 spatial_size=96, features: Sequence[int] = DEFAULT_FEATURES, dropout: float = 0.2,
                 timesteps: int = 1000, mode: str = "train", *, num_steps: int = 10, batch_max: int = 4,
                 debug_flags: int = 0, precision: str = "fp16", dual_stream: bool = True):
        super().__init__()
        if spatial_dims != 3:
            raise NotImplementedError("only spatial_dims == 3")
        _lib.load()  # fail loudly at construction if the CUDA library is missing
        self.num_classes = out_channels
        self.in_channels = in_channels
        self.mode = mode
        self.features = tuple(int(v) for v in features)
        if len(self.features) != 6:
            raise ValueError("features must have 6 entries (denoiser.py:265)")
        # window shape (spatial_size, image_size, image_size) as Engine.infer builds it (engine.py:169)
        hw = (image_size, image_size) if isinstance(image_size, int) else tuple(image_size)
        self.patch = (int(spatial_size),) + tuple(int(v) for v in hw)
        if precision not in PRECISIONS:
            raise ValueError('precision must be "fp16" (default: 11-bit mantissa operands, the reference\'s AMP precision, '
                             'test.py:104), "bf16" (8-bit mantissa, 2e-2 gate) or "fp32x3" (split-bf16 operands, 1e-4 gate; '
                             'SURVEY 8d)')
        self.num_steps, self.batch_max, self.debug_flags = int(num_steps), int(batch_max), int(debug_flags)
        self._set_precision_flags(precision)
        if dual_stream:  # batches of >= 4 windows: two half batches on two internal streams (bit-identical results)
            self.debug_flags |= _lib.DUNET_FLAG_DUAL_STREAM
        self.timesteps = timesteps
        self.schedule = DdimSchedule.build(self.num_steps, timesteps)
        holder = _Node()
        _init_like_reference(holder, in_channels, out_channels, self.features)
        # expose parameters under the reference's top-level names: embed_model.* and model.*
        self.add_module("embed_params", holder._modules["embed_model"])
        self.add_module("model_params", holder._modules["model"])
        self._register_state_dict_hook(DiffUNetB200._rename_on_save)
        self.register_load_state_dict_pre_hook(DiffUNetB200._rename_on_load)
        object.__setattr__(self, "_rt", _Runtime(self))
        object.__setattr__(self, "_emb_keepalive", None)
        object.__setattr__(self, "embed_model", EncoderB200(self))
        object.__setattr__(self, "model", DenoiserB200(self))
        object.__setattr__(self, "sample_diffusion", SampleDiffusionB200(self))
        object.__setattr__(self, "diffusion", _TrainDiffusion(timesteps))
        object.__setattr__(self, "sampler", _UniformSampler(timesteps))

    def _set_precision_flags(self, precision: str) -> None:
        self.precision = precision
        self.debug_flags &= ~(_lib.DUNET_FLAG_FP32X3 | _lib.DUNET_FLAG_FP16)
        if precision == "fp32x3":
            self.debug_flags |= _lib.DUNET_FLAG_FP32X3
        elif precision == "fp16":
            self.debug_flags |= _lib.DUNET_FLAG_FP16

    def set_precision(self, precision: str) -> "DiffUNetB200":
        """Switch the arithmetic mode of the kernels ("fp16" | "bf16" | "fp32x3"); the plan (packed weights) is rebuilt on
        the next call.  EngineB200 maps the reference's ``use_amp`` flag onto this (test.py:104,119)."""
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {PRECISIONS}")
        if precision != self.precision:
            self._set_precision_flags(precision)
            self._rt.close()
            self._rt.weights_sig = None
            self._rt.workspaces.clear()
        return self

    # ---- checkpoint keys: "embed_model.*" / "model.*" exactly like the reference ---------------------------------
    # Implemented with state-dict hooks so that it also holds when this module is a sub-module (nn.DataParallel /
    # DistributedDataParallel wrap it as ``module.``: the parent passes ``destination`` and ``prefix`` and ignores return values).
    @staticmethod
    def _rename_on_save(module, state_dict, prefix, local_metadata):
        for k in list(state_dict.keys()):
            if k.startswith(prefix + "embed_params."):
                state_dict[prefix + "embed_model." + k[len(prefix) + len("embed_params."):]] = state_dict.pop(k)
            elif k.startswith(prefix + "model_params."):
                state_dict[prefix + "model." + k[len(prefix) + len("model_params."):]] = state_dict.pop(k)
        return state_dict

    @staticmethod
    def _rename_on_load(module, state_dict, prefix, *args):
        for k in list(state_dict.keys()):
            if k.startswith(prefix + "embed_model."):
                state_dict[prefix + "embed_params." + k[len(prefix) + len("embed_model."):]] = state_dict.pop(k)
            elif k.startswith(prefix + "model."):
                state_dict[prefix + "model_params." + k[len(prefix) + len("model."):]] = state_dict.pop(k)

    def load_state_dict(self, state_dict, strict: bool = True, **kwargs):
        # checkpoints saved from nn.DataParallel / DDP carry a "module." prefix (the reference saves self.model.state_dict()
        # of the wrapped module in multi-GPU training, light_training); accept both
        if state_dict and all(k.startswith("module.") for k in state_dict):
            state_dict = type(state_dict)((k[len("module."):], v) for k, v in state_dict.items())
        return super().load_state_dict(dict(state_dict), strict=strict, **kwargs)

    def __del__(self):
        try:
            self._rt.close()
        except Exception:
            pass

    # ---- helpers -------------------------------------------------------------------------------------------------
    def _check_image(self, image: torch.Tensor):
        if image.dim() != 5 or image.shape[1] != self.in_channels or tuple(image.shape[2:]) != self.patch:
            raise ValueError(f"expected image [B, {self.in_channels}, {self.patch}], got {tuple(image.shape)}")
        if image.shape[0] > self.batch_max:
            raise ValueError(f"batch {image.shape[0]} exceeds batch_max {self.batch_max}")

    def _upload_embeddings(self, embeddings, B, ws):
        rt = self._rt
        token = (tuple(id(t) for t in embeddings), B)
        if rt.emb_token == token:
            return  # the workspace already holds exactly these tensors (produced by our own encoder)
        lib = _lib.load()
        keep = []
        for lvl, e in enumerate(embeddings):
            e = _f32c(e, f"embeddings[{lvl}]")
            keep.append(e)
            with torch.cuda.device(e.device):
                _lib.check(lib.dunet_set_embedding(rt.plan, lvl, _ptr(e), B, _ptr(ws), _stream()))
        rt.emb_token = token
        self._emb_keepalive = list(embeddings)  # ids in the token stay unique while these are alive

    def _run_ddim(self, image, noise, run_encoder=True, want_steps=False, want_final=True, acc=None, scale=1.0,
                  accumulate=False):
        rt = self._rt
        B = image.shape[0]
        plan = rt.ensure(image.device)
        ws = rt.workspace(B)
        if acc is None:
            acc = torch.empty_like(noise)
        per = torch.empty((self.num_steps,) + tuple(noise.shape), dtype=torch.float32, device=noise.device) if want_steps else None
        fin = torch.empty_like(noise) if want_final else None
        with torch.cuda.device(image.device):
            _lib.check(_lib.load().dunet_ddim_sample(plan, _ptr(image), _ptr(noise), _ptr(acc), _ptr(per), _ptr(fin), B,
                                                     1 if run_encoder else 0, ctypes.c_float(scale), 1 if accumulate else 0,
                                                     _ptr(ws), _stream()))
        if run_encoder:
            rt.emb_token = None
        return {"acc": acc, "per_step": per, "final_x": fin}

    def infer_windows(self, volume: torch.Tensor, starts, out_volume: torch.Tensor, *, noise: torch.Tensor = None,
                      seed: int = 0, noise_ids=None, ensemble: int = 1, count_volume: torch.Tensor = None,
                      weights: torch.Tensor = None) -> None:
        """One iteration of the window loop of the sliding-window driver, fused (``dunet_infer_windows``): crop the windows
        at ``starts`` ([b, 3]) out of ``volume`` ([in_channels, D, H, W] fp32, padded to >= the patch; [D, H, W] is accepted
        when in_channels == 1), run encoder + DDIM on them and do
        ``out_volume[:, window] += pred`` window by window.  Bit-identical to crop + forward(pred_type="ddim_sample") +
        ``out[slices] += pred`` (engine.py:173-177, models/diffusion/diffusion.py:86-102).  ``noise`` ([b, C, *patch] or
        [R, b, C, *patch]) fixes the initial x_T; otherwise the library draws it from (seed, noise_ids[b], draw)."""
        if not volume.is_cuda or volume.dtype != torch.float32 or not volume.is_contiguous():
            raise RuntimeError("volume must be a contiguous fp32 CUDA tensor: the B200 path has no CPU fallback")
        if not ((volume.dim() == 4 and volume.shape[0] == self.in_channels) or (volume.dim() == 3 and self.in_channels == 1)):
            raise ValueError(f"volume must be [{self.in_channels}, D, H, W]" + (" or [D, H, W]" if self.in_channels == 1 else "")
                             + f", got {tuple(volume.shape)}")
        b = len(starts)
        if b < 1 or b > self.batch_max:
            raise ValueError(f"{b} windows outside [1, batch_max = {self.batch_max}]")
        vol = tuple(volume.shape[-3:])
        if tuple(out_volume.shape) != (self.num_classes,) + vol or out_volume.dtype != torch.float32 or not out_volume.is_contiguous():
            raise ValueError(f"out_volume must be contiguous fp32 {(self.num_classes,) + vol}")
        rt = self._rt
        plan = rt.ensure(volume.device)
        ws = rt.workspace(b)
        st = (ctypes.c_int32 * (3 * b))(*[int(x) for s3 in starts for x in s3])
        ids = None
        if noise is not None:
            noise = _f32c(noise, "noise")
            if tuple(noise.shape) not in ((b, self.num_classes) + self.patch, (ensemble, b, self.num_classes) + self.patch):
                raise ValueError(f"noise must be [{ensemble}, {b}, {self.num_classes}, *{self.patch}], got {tuple(noise.shape)}")
        else:
            if noise_ids is None:
                raise ValueError("pass noise= or noise_ids= (one counter-based noise stream id per window)")
            ids = (ctypes.c_int64 * b)(*[int(i) for i in noise_ids])
        with torch.cuda.device(volume.device):
            _lib.check(_lib.load().dunet_infer_windows(plan, _ptr(volume), _lib.i32x3(vol), st, b, _ptr(noise), ctypes.c_uint64(seed & (2 ** 64 - 1)),
                                                       ids, int(ensemble), _ptr(out_volume), _ptr(count_volume), _ptr(weights),
                                                       _ptr(ws), _stream()))
        rt.emb_token = None

    # ---- the reference's Diffusion.forward dispatch (models/diffusion/diffusion.py:49-63) ------------------------
    def forward(self, image: torch.Tensor = None, x: torch.Tensor = None, step: torch.Tensor = None,
                pred_type: str = None, noise: torch.Tensor = None, ensemble: int = 1):
        if image is not None and x is not None:
            assert image.device == x.device
        if pred_type == "q_sample":
            return self.q_sample(x)
        elif pred_type == "denoise":
            return self.denoise(image, x, step)
        elif pred_type == "ddim_sample":
            return self.ddim_sample(image, noise=noise, ensemble=ensemble)
        raise NotImplementedError(f"No such prediction type : {pred_type}")

    def q_sample(self, x):
        """models/diffusion/diffusion.py:65-69: (x_t, t, noise) with t ~ UniformSampler and noise ~ N(0, 1); the noise comes
        from the library's counter-based generator, seeded from torch's global generator (torch.manual_seed applies)."""
        t, _ = self.sampler.sample(x.shape[0], x.device)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        sample, noise = self.diffusion.q_sample(x, t, None, seed=seed, return_noise=True)
        return sample, t, noise

    def denoise(self, image, x, step):
        assert image.size(0) == x.size(0) == step.size(0)
        embeddings = self.embed_model(image)
        return self.model(x=x, t=step, embeddings=embeddings, image=image)

    def ddim_sample_uncertainty(self, image: torch.Tensor, noise: torch.Tensor = None, uncer_step: int = 4) -> torch.Tensor:
        """Upstream Diff-UNet's uncertainty-weighted step fusion (SURVEY 8f-4; this reference returns the plain sum,
        models/diffusion/diffusion.py:94-98): ``uncer_step`` independent DDIM runs per window, then for every step the
        run-averaged model output gives an uncertainty map that weights the sum of the runs' clamped x0 predictions
        (``dunet_uncertainty_fuse``).  ``noise``: optional [uncer_step, B, C, *patch]."""
        image = _f32c(image, "image")
        self._check_image(image)
        B = image.shape[0]
        shape = (B, self.num_classes) + self.patch
        if noise is None:
            noise = torch.randn((uncer_step,) + shape, device=image.device)
        noise = _f32c(noise, "noise")
        if tuple(noise.shape) != (uncer_step,) + shape:
            raise ValueError(f"noise must be {(uncer_step,) + shape}, got {tuple(noise.shape)}")
        steps = torch.empty((uncer_step, self.num_steps) + shape, dtype=torch.float32, device=image.device)
        rt = self._rt
        plan = rt.ensure(image.device)
        ws = rt.workspace(B)
        scratch = torch.empty(shape, dtype=torch.float32, device=image.device)
        lib = _lib.load()
        with torch.cuda.device(image.device):
            for r in range(uncer_step):
                _lib.check(lib.dunet_ddim_sample(plan, _ptr(image), _ptr(noise[r]), _ptr(scratch), _ptr(steps[r]), None, B,
                                                 1 if r == 0 else 0, ctypes.c_float(1.0), 0, _ptr(ws), _stream()))
            out = torch.empty(shape, dtype=torch.float32, device=image.device)
            _lib.check(lib.dunet_uncertainty_fuse(_ptr(steps), uncer_step, self.num_steps, out.numel(), _ptr(out), _stream()))
        rt.emb_token = None
        return out

    def ddim_sample(self, image: torch.Tensor, noise: torch.Tensor = None, ensemble: int = 1) -> torch.Tensor:
        """Sum over the N DDIM steps of the clamped x0 prediction for every window of the batch
        (models/diffusion/diffusion.py:86-102).  ``noise`` ([B, C, *patch], or [R, B, C, *patch] with ``ensemble=R``)
        replaces the reference's internal ``randn`` draws so runs can be compared on identical noise.
        ``ensemble=R`` (BASELINE config 4; not in the reference) averages the summed outputs of R independent noise
        draws; the encoder runs once."""
        image = _f32c(image, "image")
        if image.dim() == 5 and image.shape[0] > self.batch_max:
            # more windows than the plan's batch_max (the reference accepts any sw_batch_size and loops at batch 1,
            # diffusion.py:88-89): process them in chunks -- results are identical, batching is transparent
            B = image.shape[0]
            if noise is not None:
                noise = _f32c(noise, "noise")
                noise = noise.unsqueeze(0) if noise.dim() == 5 else noise
            outs = []
            for lo in range(0, B, self.batch_max):
                hi = min(lo + self.batch_max, B)
                outs.append(self.ddim_sample(image[lo:hi], None if noise is None else noise[:, lo:hi].contiguous(), ensemble))
            return torch.cat(outs)
        self._check_image(image)
        B = image.shape[0]
        shape = (B, self.num_classes) + self.patch
        if noise is None:
            noise = torch.randn((ensemble,) + shape, device=image.device)
        noise = _f32c(noise, "noise")
        if noise.dim() == 5:
            noise = noise.unsqueeze(0)
        if tuple(noise.shape) != (ensemble,) + shape:
            raise ValueError(f"noise must be {(ensemble,) + shape} (or {shape} when ensemble == 1), got {tuple(noise.shape)}")
        acc = torch.empty(shape, dtype=torch.float32, device=image.device)
        for r in range(ensemble):
            self._run_ddim(image, noise[r], run_encoder=(r == 0), want_final=False, acc=acc, scale=1.0 / ensemble,
                           accumulate=(r > 0))
        return acc
