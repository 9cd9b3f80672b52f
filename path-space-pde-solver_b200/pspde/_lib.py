"""ctypes binding of libpspde.so (C ABI: include/pspde.h).

The product path requires the CUDA library: ``load()`` raises if ``libpspde.so`` has not been built or no CUDA
device is present -- there is no CPU fallback.  (``bind(path)`` only attaches prototypes to an already chosen
shared object; tests use it to drive the host-side emulator build of the same sources.)
"""
import ctypes
import os

PSPDE_MAX_LAYERS = 4
PROBLEM_OU, PROBLEM_DW, PROBLEM_HEAT, PROBLEM_ALLEN_CAHN = 0, 1, 2, 3
FLAG_DENSE_AB = 1
NET_DENSENET, NET_MLP_TANH = 0, 1
TIME_FIRST, TIME_NONE, TIME_LAST = 0, 1, 2
NOISE_INJECT, NOISE_PHILOX = 0, 1
DOMAIN_SPHERE, DOMAIN_BOX, DOMAIN_ANNULUS = 1, 2, 3
H_ZERO, H_EXP_LINEAR, H_EXP_NONLINEAR, H_EXP_NONLINEAR_SIN, H_HELMHOLTZ, H_COMMITTOR = 0, 1, 2, 3, 4, 6
ABI_VERSION = 3

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpspde.so")


class pspde_cfg(ctypes.Structure):
    _fields_ = [
        ("K_local", ctypes.c_int32), ("k_offset", ctypes.c_int32), ("d", ctypes.c_int32), ("N", ctypes.c_int32),
        ("dt", ctypes.c_float),
        ("problem_id", ctypes.c_int32), ("problem_flags", ctypes.c_int32),
        ("net_id", ctypes.c_int32), ("n_layers", ctypes.c_int32),
        ("dims", ctypes.c_int32 * (PSPDE_MAX_LAYERS + 1)),
        ("time_mode", ctypes.c_int32), ("adaptive", ctypes.c_int32), ("noise_mode", ctypes.c_int32),
        ("x0_per_path", ctypes.c_int32),
        ("seed", ctypes.c_uint64), ("offset", ctypes.c_uint32), ("n_sets", ctypes.c_int32),
        ("xi_stride_k", ctypes.c_int64), ("xi_stride_j", ctypes.c_int64), ("xi_stride_n", ctypes.c_int64),
        ("d_abs_max", ctypes.c_float),
    ]


class pspde_udiag(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int32), ("nx1", ctypes.c_int32), ("d1", ctypes.c_int32), ("xb", ctypes.c_float),
                ("dx", ctypes.c_float), ("table", ctypes.c_void_p), ("uL2", ctypes.c_void_p), ("quirk_path", ctypes.c_int32)]


class pspde_elliptic(ctypes.Structure):
    _fields_ = [("domain", ctypes.c_int32), ("radius", ctypes.c_float), ("x_l", ctypes.c_float),
                ("x_r", ctypes.c_float), ("one_boundary", ctypes.c_int32), ("h_id", ctypes.c_int32),
                ("h_param", ctypes.c_float * 3), ("radius_in", ctypes.c_float)]


class pspde_ensemble(ctypes.Structure):
    _fields_ = [("n_models", ctypes.c_int32), ("seeds", ctypes.c_void_p), ("theta_stride", ctypes.c_int64),
                ("x0_stride", ctypes.c_int64)]


class pspde_adam_member(ctypes.Structure):
    _fields_ = [("lr_over_bc1", ctypes.c_float), ("sqrt_bc2", ctypes.c_float), ("one_minus_beta1", ctypes.c_float),
                ("beta2", ctypes.c_float), ("one_minus_beta2", ctypes.c_float), ("eps", ctypes.c_float),
                ("step", ctypes.c_int32), ("reserved", ctypes.c_int32)]


_P = ctypes.c_void_p
_CFG = ctypes.POINTER(pspde_cfg)
_ENS = ctypes.POINTER(pspde_ensemble)
_ELL = ctypes.POINTER(pspde_elliptic)

PROTOTYPES = {
    "pspde_abi_version": (ctypes.c_int, []),
    "pspde_last_error": (ctypes.c_char_p, []),
    "pspde_launch_count": (ctypes.c_uint64, []),
    "pspde_set_profile_buffer": (None, [_P]),
    "pspde_theta_size": (ctypes.c_int64, [_CFG]),
    "pspde_workspace_bytes": (ctypes.c_size_t, [_CFG]),
    "pspde_workspace_bytes_fwd": (ctypes.c_size_t, [_CFG]),
    "pspde_rollout_fwd": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_rollout_fwd_diag": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.POINTER(pspde_udiag),
                                              _P, ctypes.c_size_t, _P]),
    "pspde_rollout_bwd_detached": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_grad_from_ckpt": (ctypes.c_int, [_CFG, _P, _P, ctypes.c_int, ctypes.c_int, _P, _P, ctypes.c_size_t, _P]),
    "pspde_fwd_ckpt_bytes": (ctypes.c_size_t, [_CFG]),
    "pspde_rollout_fwd_ckpt": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.POINTER(pspde_udiag),
                                              _P, ctypes.c_size_t, _P, ctypes.c_size_t, _P]),
    "pspde_grad_from_fwd_ckpt": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, ctypes.c_size_t, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_rollout_attached": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, ctypes.c_float, _P, _P, _P, _P, _P, _P, _P,
                                              _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_rollout_attached_diag": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, ctypes.c_float, _P, _P, _P, _P, _P, _P, _P,
                                                   _P, ctypes.POINTER(pspde_udiag), _P, _P, ctypes.c_size_t, _P]),
    "pspde_importance_sampling": (ctypes.c_int, [_CFG, _P, _P, _P, _P, _P, ctypes.c_float, _P, _P, _P, _P, _P,
                                                 ctypes.c_size_t, _P]),
    "pspde_philox_dump": (ctypes.c_int, [_CFG, _P, _P]),
    "pspde_diffusion_workspace_bytes": (ctypes.c_size_t, [_CFG, ctypes.c_float]),
    "pspde_diffusion_fwd": (ctypes.c_int, [_CFG, ctypes.c_float, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                           ctypes.c_size_t, _P]),
    "pspde_diffusion_bwd": (ctypes.c_int, [_CFG, ctypes.c_float, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                           ctypes.c_size_t, _P]),
    "pspde_elliptic_workspace_bytes": (ctypes.c_size_t, [_CFG, _ELL]),
    "pspde_elliptic_fwd": (ctypes.c_int, [_CFG, _ELL, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_elliptic_bwd": (ctypes.c_int, [_CFG, _ELL, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_diffusion_sample": (ctypes.c_int, [_CFG, ctypes.c_float, ctypes.c_float, _P, _P, _P]),
    "pspde_tc_selftest": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _P, _P, _P, _P]),
    "pspde_tma_selftest": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _P, _P, _P, _P]),
    "pspde_mma_probe": (ctypes.c_int, [ctypes.c_int, _P, _P]),
    "pspde_lv_cotangents": (ctypes.c_int, [ctypes.c_int, ctypes.c_double, ctypes.c_int, _P, _P, _P, _P, _P, _P]),
    "pspde_adam_flat": (ctypes.c_int, [ctypes.c_int64, _P, _P, _P, _P, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                       ctypes.c_double, ctypes.c_int64, _P]),
    "pspde_ensemble_workspace_bytes": (ctypes.c_size_t, [_CFG, _ENS]),
    "pspde_ensemble_fwd": (ctypes.c_int, [_CFG, _ENS, _P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.POINTER(pspde_udiag),
                                          _P, ctypes.c_size_t, _P]),
    "pspde_ensemble_bwd_detached": (ctypes.c_int, [_CFG, _ENS, _P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "pspde_ensemble_lv_cotangents": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int, ctypes.c_double, ctypes.c_int, _P, _P, _P,
                                                    _P, _P, _P]),
    "pspde_adam_member_make": (ctypes.c_int, [ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                              ctypes.c_int64, ctypes.POINTER(pspde_adam_member)]),
    "pspde_ensemble_adam": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, _P, _P, _P, _P, _P, _P]),
    "pspde_fma_probe": (ctypes.c_int64, [ctypes.c_int, _P, _P]),
    "pspde_fma_probe_ex": (ctypes.c_int64, [ctypes.c_int, ctypes.c_int, _P, _P]),
}


def bind(path):
    """dlopen `path` and attach the prototypes of include/pspde.h; raises if a symbol is missing."""
    lib = ctypes.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError -> the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    if lib.pspde_abi_version() != ABI_VERSION:
        raise RuntimeError("libpspde ABI %d != binding %d" % (lib.pspde_abi_version(), ABI_VERSION))
    return lib


_lib = None


def load():
    """The CUDA library; raises (never falls back) when it is missing or CUDA is unavailable."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s not built: run `python __graft_entry__.py` (build()) first" % LIB_PATH)
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("pspde needs a CUDA device (B200 / sm_100a); there is no CPU fallback")
        _lib = bind(LIB_PATH)
    return _lib


def check(lib, rc):
    if rc != 0:
        raise RuntimeError("libpspde error %d: %s" % (rc, lib.pspde_last_error().decode()))


def make_cfg(K_local, d, N, dt, problem_id, net_id, dims, time_mode, adaptive=True, k_offset=0, problem_flags=0,
             noise_mode=NOISE_PHILOX, seed=0, offset=0, x0_per_path=False, xi_strides=(0, 0, 0), n_sets=0,
             d_abs_max=0.0):
    c = pspde_cfg()
    c.K_local, c.k_offset, c.d, c.N = int(K_local), int(k_offset), int(d), int(N)
    c.dt = float(dt)
    c.problem_id, c.problem_flags = int(problem_id), int(problem_flags)
    c.net_id, c.n_layers = int(net_id), len(dims) - 1
    if len(dims) - 1 > PSPDE_MAX_LAYERS:
        raise NotImplementedError("networks with more than %d linear layers are not supported" % PSPDE_MAX_LAYERS)
    for i, v in enumerate(dims):
        c.dims[i] = int(v)
    c.time_mode, c.adaptive, c.noise_mode = int(time_mode), int(bool(adaptive)), int(noise_mode)
    c.x0_per_path = int(bool(x0_per_path))
    c.seed, c.offset = int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 32 - 1)
    c.n_sets = int(n_sets)
    c.xi_stride_k, c.xi_stride_j, c.xi_stride_n = (int(s) for s in xi_strides)
    c.d_abs_max = float(d_abs_max)
    return c


def make_elliptic(domain, radius=1.0, x_l=-1.0, x_r=1.0, one_boundary=False, h_id=H_ZERO, h_param=(0.0, 0.0, 0.0),
                  radius_in=0.0):
    e = pspde_elliptic()
    e.domain, e.radius, e.x_l, e.x_r = int(domain), float(radius), float(x_l), float(x_r)
    e.one_boundary, e.h_id, e.radius_in = int(bool(one_boundary)), int(h_id), float(radius_in)
    for i in range(3):
        e.h_param[i] = float(h_param[i]) if i < len(h_param) else 0.0
    return e
