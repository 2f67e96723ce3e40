"""unet.cu_b200 -- Python host-side mirror of the C ABI in include/unet_b200.h (ctypes, no torch types in any
signature).  The shared library is built in-tree by `__graft_entry__.build()` / `make -C unet.cu_b200`.

The package fails loudly when the CUDA extension is missing: there is no CPU fallback.

Because the directory name contains a dot it is loaded with importlib (see __graft_entry__.load_package()).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# UB_LIB_VARIANT=<name> loads lib/libunet_b200_<name>.so: a development switch for A/B-measuring compile-time kernel
# variants in one GPU session (unet.cu_b200/Makefile, VARIANT=).  Unset = the shipped library.
_VARIANT = os.environ.get("UB_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, "lib", f"libunet_b200{'_' + _VARIANT if _VARIANT else ''}.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "unet_b200.h")

UB_NCCL_ID_BYTES = 128


class UbConfig(C.Structure):
    """UbConfig of include/unet_b200.h (UnetConfig of train_unet.cu:3318-3336, generalised)."""
    _fields_ = [("B", C.c_int), ("C_in", C.c_int), ("C_model", C.c_int), ("C_out", C.c_int), ("H", C.c_int),
                ("W", C.c_int), ("max_period", C.c_int), ("n_levels", C.c_int), ("channel_mult", C.c_int * 8),
                ("n_res_blocks", C.c_int), ("att_start_level", C.c_int), ("head_size", C.c_int),
                ("gn_n_groups", C.c_int), ("n_timesteps", C.c_int), ("seed", C.c_ulonglong),
                ("use_cuda_graph", C.c_int), ("compute_dinput", C.c_int), ("random_flip", C.c_int),
                ("num_classes", C.c_int), ("ema_rate", C.c_float), ("resblock_updown", C.c_int),
                ("use_scale_shift_norm", C.c_int), ("dropout", C.c_float), ("super_res", C.c_int),
                ("learn_sigma", C.c_int), ("noise_schedule", C.c_int), ("class_dropout", C.c_float)]


class UbConvSeg(C.Structure):
    """UbConvSeg of include/unet_b200.h: one input of ub_conv2d_nhwc_fused (NHWC bf16, channel pitch ldx) and its
    packed weights."""
    _fields_ = [("x_bf16", C.c_void_p), ("C_in", C.c_int), ("ldx", C.c_int), ("w_bf16", C.c_void_p),
                ("ksize", C.c_int)]


class UbConvEpilogue(C.Structure):
    """UbConvEpilogue of include/unet_b200.h: the conv kernels' epilogue (bias, second bias, per-image row, residual,
    output layout, GroupNorm statistics / gn-bwd hooks)."""
    _fields_ = [("bias", C.c_void_p), ("bias2", C.c_void_p), ("rowvec", C.c_void_p), ("residual_bf16", C.c_void_p),
                ("ldr", C.c_int), ("out", C.c_void_p), ("ldo", C.c_int), ("out_mode", C.c_int),
                ("stats", C.c_void_p), ("gn_x_bf16", C.c_void_p), ("gn_ldx", C.c_int), ("gn_chsum", C.c_void_p),
                ("gn_gamma", C.c_void_p), ("gn_beta", C.c_void_p), ("gn_S", C.c_void_p), ("gn_silu", C.c_int),
                ("gn_groups", C.c_int)]


class UbConvPlanInfo(C.Structure):
    """UbConvPlanInfo of include/unet_b200.h: the plan ub_conv2d_nhwc_fused launched (or stopped at)."""
    _fields_ = [(n, C.c_int) for n in ("kernel", "BN", "nacc", "ms", "stages", "w_resident", "TW", "TH", "TB", "grid")]


UB_KINDS = ("conv_igemm", "wgrad_igemm", "groupnorm", "attention", "eltwise", "small", "optimizer")


class UbProfile(C.Structure):
    _fields_ = [("ms", C.c_double * 7), ("flops", C.c_double * 7), ("bytes", C.c_double * 7),
                ("launches", C.c_int * 7), ("total_ms", C.c_double)]


class UbError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load libunet_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise UbError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the CUDA extension is mandatory, there is no CPU path)")
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _declare(_lib)
    return _lib


def _declare(L: C.CDLL) -> None:
    fp, vp, i = C.c_void_p, C.c_void_p, C.c_int
    L.ub_last_error.restype = C.c_char_p
    L.ub_version.restype = C.c_char_p
    L.ub_launch_count.restype = C.c_ulonglong
    L.ub_set_stream.argtypes = [vp]
    L.ub_default_config.argtypes = [C.POINTER(UbConfig)]
    L.ub_default_config.restype = None
    L.ub_num_params.argtypes = [C.POINTER(UbConfig)]
    L.ub_num_params.restype = C.c_size_t
    L.ub_trainer_create.argtypes = [C.POINTER(vp), C.POINTER(UbConfig), i]
    L.ub_trainer_destroy.argtypes = [vp]
    L.ub_trainer_destroy.restype = None
    L.ub_trainer_load.argtypes = [vp, C.c_char_p]
    L.ub_trainer_save.argtypes = [vp, C.c_char_p, i]
    L.ub_read_checkpoint_header.argtypes = [C.c_char_p, C.POINTER(UbConfig)]
    L.ub_trainer_save_ema.argtypes = [vp, C.c_char_p]
    L.ub_trainer_set_labels.argtypes = [vp, vp, C.c_size_t]
    L.ub_trainer_get_dropout_mask.argtypes = [vp, i, vp, C.c_size_t]
    for n in ("set_params", "get_params", "get_grads", "get_output", "get_batch", "get_dinput", "get_ema", "set_ema",
              "set_low_res", "get_cond"):
        getattr(L, "ub_trainer_" + n).argtypes = [vp, fp, C.c_size_t]
    L.ub_trainer_forward_backward.argtypes = [vp, fp, fp, fp, C.POINTER(C.c_float)]
    L.ub_trainer_update.argtypes = [vp] + [C.c_float] * 5
    L.ub_trainer_train_step.argtypes = [vp, fp, fp, fp] + [C.c_float] * 5 + [C.POINTER(C.c_float)]
    L.ub_trainer_train_step_device.argtypes = [vp, fp] + [C.c_float] * 5
    L.ub_trainer_set_next_batch.argtypes = [vp, vp]
    L.ub_trainer_sync.argtypes = [vp]
    L.ub_trainer_last_loss.argtypes = [vp, C.POINTER(C.c_float)]
    L.ub_trainer_last_loss_terms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.ub_trainer_set_step.argtypes = [vp, i]
    L.ub_trainer_get_flips.argtypes = [vp, vp, C.c_size_t]
    L.ub_trainer_get_effective_labels.argtypes = [vp, vp, C.c_size_t]
    L.ub_trainer_set_guidance.argtypes = [vp, C.c_float]
    L.ub_set_layer_precision.argtypes = [i]
    L.ub_groupnorm_nhwc_forward.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, i, i, i]
    L.ub_groupnorm_nhwc_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i]
    L.ub_groupnorm_nhwc_backward_apply.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i]
    L.ub_conv2d_nhwc_fused.argtypes = [C.POINTER(UbConvSeg), i, i, i, i, i, C.POINTER(UbConvEpilogue), i,
                                       C.POINTER(UbConvPlanInfo)]
    L.ub_conv2d_nhwc_wgrad_acc.argtypes = [vp, i, vp, i, vp, vp, vp, i, i, i, i, i, i, C.POINTER(i), C.POINTER(i)]
    L.ub_pack_conv_weight.argtypes = [vp, vp, vp, i, i, i]
    L.ub_trainer_stream.argtypes = [vp]
    L.ub_trainer_stream.restype = vp
    L.ub_trainer_launches_per_step.argtypes = [vp]
    L.ub_trainer_predict.argtypes = [vp, fp, fp, fp]
    L.ub_trainer_profile.argtypes = [vp, i, C.POINTER(UbProfile)]
    L.ub_trainer_sample.argtypes = [vp, fp, i, i, fp, C.c_ulonglong, fp]
    L.ub_space_timesteps.argtypes = [i, C.c_char_p, vp, i]
    L.ub_beta_schedule.argtypes = [i, i, vp]
    L.ub_trainer_sample_spaced.argtypes = [vp, vp, i, i, C.c_float, i, fp, fp, C.c_ulonglong, fp]
    L.ub_dataloader_open.argtypes = [C.POINTER(vp), C.c_char_p, i, i, i]
    L.ub_dataloader_info.argtypes = [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(i),
                                     C.POINTER(C.c_longlong)]
    L.ub_dataloader_next.argtypes = [vp]
    L.ub_dataloader_next.restype = vp
    L.ub_dataloader_reset.argtypes = [vp]
    L.ub_dataloader_reset.restype = None
    L.ub_dataloader_close.argtypes = [vp]
    L.ub_dataloader_close.restype = None
    L.ub_nccl_get_unique_id.argtypes = [vp]
    L.ub_trainer_attach_dp.argtypes = [vp, i, i, vp, i]


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise UbError(f"{what} failed with code {rc}: {lib().ub_last_error().decode()}")


def default_config(**over) -> UbConfig:
    cfg = UbConfig()
    lib().ub_default_config(C.byref(cfg))
    for k, v in over.items():
        if k == "channel_mult":
            for j, m in enumerate(v):
                cfg.channel_mult[j] = int(m)
            cfg.n_levels = len(v)
        else:
            setattr(cfg, k, v)
    return cfg


def num_params(cfg: UbConfig) -> int:
    return int(lib().ub_num_params(C.byref(cfg)))


def space_timesteps(n_timesteps: int, spec: str) -> list[int]:
    """guided-diffusion respace.space_timesteps as a sorted list: "ddimN" or comma-separated section counts ("250",
    "10,10,10"); raises UbError for a malformed or unsatisfiable spec.  Needs no GPU."""
    out = np.empty(max(int(n_timesteps), 1), dtype=np.int32)
    n = lib().ub_space_timesteps(int(n_timesteps), spec.encode(), out.ctypes.data_as(C.c_void_p), out.size)
    if n < 0:
        check(n, "space_timesteps")
    return [int(v) for v in out[:n]]


UB_SCHEDULE_LINEAR, UB_SCHEDULE_COSINE = 0, 1
UB_SCHEDULES = {"linear": UB_SCHEDULE_LINEAR, "cosine": UB_SCHEDULE_COSINE}


def beta_schedule(schedule, n_timesteps: int) -> np.ndarray:
    """guided-diffusion's get_named_beta_schedule: the float64 betas the trainer builds its tables from, for a
    UbConfig.noise_schedule value or its name ("linear", "cosine"); raises UbError for an unknown schedule or
    n_timesteps < 1.  Needs no GPU."""
    code = UB_SCHEDULES.get(schedule, -1) if isinstance(schedule, str) else int(schedule)
    out = np.empty(max(int(n_timesteps), 1), dtype=np.float64)
    check(lib().ub_beta_schedule(code, int(n_timesteps), out.ctypes.data_as(C.c_void_p)), "beta_schedule")
    return out


UB_SAMPLERS = {"ddim": 0, "ancestral": 1}


def _ptr(a: Optional[np.ndarray]):
    if a is None:
        return None
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


class Trainer:
    """Mirror of the train_unet.cu loop body (train_unet.cu:5019-5037) over host (numpy) buffers."""

    def __init__(self, cfg: Optional[UbConfig] = None, device: int = 0, **over):
        self.cfg = cfg if cfg is not None else default_config(**over)
        self._h = C.c_void_p()
        check(lib().ub_trainer_create(C.byref(self._h), C.byref(self.cfg), device), "ub_trainer_create")
        self.nparams = num_params(self.cfg)

    def close(self):
        if self._h:
            lib().ub_trainer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- parameters / checkpoints
    def set_params(self, flat: np.ndarray):
        flat = np.ascontiguousarray(flat, dtype=np.float32)
        check(lib().ub_trainer_set_params(self._h, _ptr(flat), flat.size), "set_params")

    def _get(self, fn, n):
        out = np.empty(n, dtype=np.float32)
        check(fn(self._h, _ptr(out), out.size), fn.__name__)
        return out

    def get_params(self):
        return self._get(lib().ub_trainer_get_params, self.nparams)

    def get_grads(self):
        return self._get(lib().ub_trainer_get_grads, self.nparams)

    def get_ema(self):
        """Moving average of the parameters (cfg.ema_rate > 0; guided-diffusion update_ema, train_unet.py:708)."""
        return self._get(lib().ub_trainer_get_ema, self.nparams)

    def set_ema(self, flat: np.ndarray):
        flat = np.ascontiguousarray(flat, dtype=np.float32)
        check(lib().ub_trainer_set_ema(self._h, _ptr(flat), flat.size), "set_ema")

    def save_ema(self, path: str):
        check(lib().ub_trainer_save_ema(self._h, path.encode()), "ub_trainer_save_ema")

    def set_labels(self, y):
        """Class labels of the batches that follow (cfg.num_classes > 0; `y` of UNetModel.forward, dev/unet.py:301-303);
        with cfg.class_dropout > 0, -1 stands for the null class."""
        y = np.ascontiguousarray(y, dtype=np.int32).reshape(-1)
        check(lib().ub_trainer_set_labels(self._h, y.ctypes.data_as(C.c_void_p), y.size), "set_labels")

    def get_effective_labels(self) -> np.ndarray:
        """The labels the last training step of a classifier-free guidance model (cfg.class_dropout > 0) used, with -1
        where it dropped the label or the caller passed -1."""
        out = np.empty(self.cfg.B, dtype=np.int32)
        check(lib().ub_trainer_get_effective_labels(self._h, out.ctypes.data_as(C.c_void_p), out.size),
              "get_effective_labels")
        return out

    def set_guidance(self, scale: float):
        """Classifier-free guidance scale of sample_spaced (GLIDE's guidance_scale: 1 = conditional, the default; 0 =
        unconditional; Ho & Salimans' w = scale - 1); needs cfg.class_dropout > 0."""
        check(lib().ub_trainer_set_guidance(self._h, float(scale)), "set_guidance")

    def get_dropout_mask(self, block: int, C_: int, H: int, W: int) -> np.ndarray:
        """Keep-mask (B, C, H, W) of 0 / 1 the last training step applied in ResBlock `block` (cfg.dropout > 0)."""
        out = np.empty((self.cfg.B, H, W, C_), dtype=np.uint8)
        check(lib().ub_trainer_get_dropout_mask(self._h, block, out.ctypes.data_as(C.c_void_p), out.size), "dropout mask")
        return np.ascontiguousarray(out.transpose(0, 3, 1, 2))

    def get_dinput(self):
        c = self.cfg
        return self._get(lib().ub_trainer_get_dinput, c.B * c.C_in * c.H * c.W).reshape(c.B, c.C_in, c.H, c.W)

    def set_low_res(self, low_res):
        """Low-res images (B, C_in, H/f, W/f) in [-1, 1] that predict / sample / sample_spaced of a super-resolution
        model (super_res = f) condition on until set again (super_res_sample.py's `low_res`)."""
        low_res = np.ascontiguousarray(low_res, dtype=np.float32)
        check(lib().ub_trainer_set_low_res(self._h, _ptr(low_res), low_res.size), "set_low_res")

    def get_cond(self) -> np.ndarray:
        """The conditioning channels (B, C_in, H, W) the last forward pass of a super-resolution model read."""
        c = self.cfg
        return self._get(lib().ub_trainer_get_cond, c.B * c.C_in * c.H * c.W).reshape(c.B, c.C_in, c.H, c.W)

    def get_flips(self) -> np.ndarray:
        """0 / 1 per image: the random horizontal flips of the last step (cfg.random_flip, train_unet.py:531-532)."""
        out = np.empty(self.cfg.B, dtype=np.int32)
        check(lib().ub_trainer_get_flips(self._h, out.ctypes.data_as(C.c_void_p), out.size), "get_flips")
        return out

    def get_batch(self):
        """The x0 batch the last step consumed, as it sits on the device (B, C_in, H, W)."""
        c = self.cfg
        return self._get(lib().ub_trainer_get_batch, c.B * c.C_in * c.H * c.W).reshape(c.B, c.C_in, c.H, c.W)

    def _out_channels(self) -> int:
        """Channels of the model output: C_out, or 2 * C_out [eps | v] for a learned-variance model."""
        return self.cfg.C_out * (2 if self.cfg.learn_sigma else 1)

    def get_output(self):
        c, co = self.cfg, self._out_channels()
        return self._get(lib().ub_trainer_get_output, c.B * co * c.H * c.W).reshape(c.B, co, c.H, c.W)

    def load(self, path: str):
        check(lib().ub_trainer_load(self._h, path.encode()), "ub_trainer_load")

    def save(self, path: str, with_adamw: bool = False):
        check(lib().ub_trainer_save(self._h, path.encode(), int(with_adamw)), "ub_trainer_save")

    # -- steps
    def forward_backward(self, x0, t=None, noise=None) -> float:
        loss = C.c_float()
        x0 = np.ascontiguousarray(x0, dtype=np.float32)
        t = None if t is None else np.ascontiguousarray(t, dtype=np.float32).reshape(-1)
        noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float32)
        check(lib().ub_trainer_forward_backward(self._h, _ptr(x0), _ptr(t), _ptr(noise), C.byref(loss)),
              "forward_backward")
        return float(loss.value)

    def update(self, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0):
        check(lib().ub_trainer_update(self._h, lr, beta1, beta2, eps, weight_decay), "update")

    def train_step(self, x0, t=None, noise=None, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
                   want_loss=True) -> Optional[float]:
        loss = C.c_float()
        x0 = np.ascontiguousarray(x0, dtype=np.float32)
        t = None if t is None else np.ascontiguousarray(t, dtype=np.float32).reshape(-1)
        noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float32)
        check(lib().ub_trainer_train_step(self._h, _ptr(x0), _ptr(t), _ptr(noise), lr, beta1, beta2, eps,
                                          weight_decay, C.byref(loss) if want_loss else None), "train_step")
        return float(loss.value) if want_loss else None

    def train_step_ptr(self, x0_host_ptr: int, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
                       loss_ref=None):
        """Same as train_step with a raw (e.g. pinned) host pointer; device-side timestep/noise draws."""
        check(lib().ub_trainer_train_step(self._h, C.c_void_p(x0_host_ptr), None, None, lr, beta1, beta2, eps,
                                          weight_decay, loss_ref), "train_step")

    def set_next_batch(self, next_x0_host_ptr: int):
        """Announce the (pinned) host batch of the NEXT train_step: its H2D copy overlaps the step that follows this call."""
        check(lib().ub_trainer_set_next_batch(self._h, C.c_void_p(next_x0_host_ptr)), "set_next_batch")

    def train_step_device(self, x0_dev_ptr: int, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0):
        check(lib().ub_trainer_train_step_device(self._h, C.c_void_p(x0_dev_ptr), lr, beta1, beta2, eps,
                                                 weight_decay), "train_step_device")

    def sync(self):
        check(lib().ub_trainer_sync(self._h), "sync")

    def last_loss(self) -> float:
        loss = C.c_float()
        check(lib().ub_trainer_last_loss(self._h, C.byref(loss)), "last_loss")
        return float(loss.value)

    def last_loss_terms(self) -> tuple:
        """(mse, vb) batch means of the last step; vb is the rescaled variational-bound term of a learned-variance
        model (learn_sigma; 0 otherwise) and last_loss() their sum."""
        mse, vb = C.c_float(), C.c_float()
        check(lib().ub_trainer_last_loss_terms(self._h, C.byref(mse), C.byref(vb)), "last_loss_terms")
        return float(mse.value), float(vb.value)

    def stream(self) -> int:
        return int(lib().ub_trainer_stream(self._h) or 0)

    def launches_per_step(self) -> int:
        return int(lib().ub_trainer_launches_per_step(self._h))

    def profile(self, reps: int = 3) -> dict:
        """Per-kernel-class device time of one step (CUDA events around every launch)."""
        p = UbProfile()
        check(lib().ub_trainer_profile(self._h, reps, C.byref(p)), "profile")
        return {k: {"ms": p.ms[j], "flops": p.flops[j], "bytes": p.bytes[j], "launches": p.launches[j]}
                for j, k in enumerate(UB_KINDS)} | {"total_ms": p.total_ms}

    def predict(self, xt, t):
        c = self.cfg
        xt = np.ascontiguousarray(xt, dtype=np.float32)
        t = np.ascontiguousarray(t, dtype=np.float32).reshape(-1)
        out = np.empty((c.B, self._out_channels(), c.H, c.W), dtype=np.float32)
        check(lib().ub_trainer_predict(self._h, _ptr(xt), _ptr(t), _ptr(out)), "predict")
        return out

    # -- data parallel
    def sample(self, x_init=None, t_start: int = -1, t_end: int = -1, noises=None, seed: int = 0) -> np.ndarray:
        """DDPM ancestral sampling (generate.py:29-79) of B images; noises: (iterations, B, C, H, W) or None."""
        c = self.cfg
        x_init = None if x_init is None else np.ascontiguousarray(x_init, dtype=np.float32)
        noises = None if noises is None else np.ascontiguousarray(noises, dtype=np.float32)
        out = np.empty((c.B, c.C_in, c.H, c.W), dtype=np.float32)
        check(lib().ub_trainer_sample(self._h, _ptr(x_init), t_start, t_end, _ptr(noises), seed, _ptr(out)), "sample")
        return out

    def sample_spaced(self, x_init=None, timesteps: Sequence[int] = (), sampler: str = "ddim", eta: float = 0.0,
                      clip_denoised: bool = True, noises=None, seed: int = 0) -> np.ndarray:
        """guided-diffusion sampling over the kept `timesteps` (ascending, e.g. space_timesteps(1000, "ddim50")):
        sampler "ddim" (ddim_sample_loop, eta in [0, 1]) or "ancestral" (p_sample_loop, fixed-large variance).
        noises: (len(timesteps), B, C, H, W), largest timestep first, or None (device draws from `seed`)."""
        if sampler not in UB_SAMPLERS:
            raise UbError(f"sampler must be one of {sorted(UB_SAMPLERS)}, got {sampler!r}")
        c = self.cfg
        ts = np.ascontiguousarray(timesteps, dtype=np.int32).reshape(-1)
        x_init = None if x_init is None else np.ascontiguousarray(x_init, dtype=np.float32)
        noises = None if noises is None else np.ascontiguousarray(noises, dtype=np.float32)
        img = c.B * c.C_in * c.H * c.W
        if (x_init is not None and x_init.size != img) or (noises is not None and noises.size != ts.size * img):
            raise UbError(f"x_init must hold {img} values and noises {ts.size} x {img}")
        out = np.empty((c.B, c.C_in, c.H, c.W), dtype=np.float32)
        check(lib().ub_trainer_sample_spaced(self._h, ts.ctypes.data_as(C.c_void_p), ts.size, UB_SAMPLERS[sampler],
                                             float(eta), int(bool(clip_denoised)), _ptr(x_init), _ptr(noises), seed,
                                             _ptr(out)), "sample_spaced")
        return out

    def attach_dp(self, rank: int, world: int, nccl_id: bytes, n_buckets: int = 0):
        buf = C.create_string_buffer(nccl_id, UB_NCCL_ID_BYTES)
        check(lib().ub_trainer_attach_dp(self._h, rank, world, buf, n_buckets), "attach_dp")


class DataLoader:
    """prepare_data.py-format reader with background prefetch (mirror of DataLoader, train_unet.cu:3035-3099)."""

    def __init__(self, path: str, B: int, rank: int = 0, world: int = 1):
        self._h = C.c_void_p()
        check(lib().ub_dataloader_open(C.byref(self._h), path.encode(), B, rank, world), "ub_dataloader_open")
        n, c, h, w, nb = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_longlong()
        lib().ub_dataloader_info(self._h, C.byref(n), C.byref(c), C.byref(h), C.byref(w), C.byref(nb))
        self.B, self.n_imgs, self.shape, self.batches_per_epoch = B, n.value, (c.value, h.value, w.value), nb.value

    def next_ptr(self) -> int:
        """Address of the (page-locked) buffer holding the next batch; valid until the call after the following one."""
        p = lib().ub_dataloader_next(self._h)
        if not p:
            raise UbError("ub_dataloader_next failed: " + lib().ub_last_error().decode())
        return p

    def next(self) -> np.ndarray:
        n = self.B * int(np.prod(self.shape))
        buf = (C.c_float * n).from_address(self.next_ptr())
        return np.frombuffer(buf, dtype=np.float32).reshape((self.B,) + self.shape).copy()

    def reset(self):
        lib().ub_dataloader_reset(self._h)

    def close(self):
        if self._h:
            lib().ub_dataloader_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(UB_NCCL_ID_BYTES)
    check(lib().ub_nccl_get_unique_id(buf), "ub_nccl_get_unique_id")
    return buf.raw


def shard_batch(global_batch: int, rank: int, world: int):
    """Contiguous batch shard of rank `rank` (SURVEY.md section 8e): samples [r*Bg/R, (r+1)*Bg/R)."""
    if global_batch % world:
        raise ValueError("global batch must be divisible by the world size")
    per = global_batch // world
    return rank * per, (rank + 1) * per
