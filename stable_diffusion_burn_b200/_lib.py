"""ctypes binding of libsdb200.so (the C ABI declared in include/sdb200.h).

The library is built in-tree by `make -C stable_diffusion_burn_b200/csrc` (see __graft_entry__.build).
There is no fallback: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsdb200.so")

_f32p = C.POINTER(C.c_float)
_u8p = C.POINTER(C.c_uint8)
_i64p = C.POINTER(C.c_int64)
_ctx = C.c_void_p

# (name, restype, argtypes) — every symbol declared in include/sdb200.h
SIGNATURES = [
    ("sdb_create", C.c_int, [C.c_int, C.POINTER(_ctx)]),
    ("sdb_destroy", C.c_int, [_ctx]),
    ("sdb_last_error", C.c_char_p, [_ctx]),
    ("sdb_version", C.c_char_p, []),
    ("sdb_tensor_count", C.c_int, [_ctx]),
    ("sdb_tensor_info", C.c_int, [_ctx, C.c_int, C.POINTER(C.c_char_p), _i64p, C.POINTER(C.c_int)]),
    ("sdb_set_tensor", C.c_int, [_ctx, C.c_char_p, _f32p, _i64p, C.c_int]),
    ("sdb_get_tensor", C.c_int, [_ctx, C.c_char_p, _f32p, C.c_int64]),
    ("sdb_init_synthetic", C.c_int, [_ctx, C.c_uint32]),
    ("sdb_weight_arena", C.c_int, [_ctx, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    ("sdb_finalize_weights", C.c_int, [_ctx]),
    ("sdb_unet_forward", C.c_int, [_ctx, _f32p, C.c_int32, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_decode_latent", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_sample_latent", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_double, C.c_int, _f32p,
                                    C.c_uint64, C.c_int, C.c_int, _f32p]),
    ("sdb_latent_to_image", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, C.c_int, _u8p]),
    ("sdb_sample_image", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_double, C.c_int, _f32p,
                                   C.c_uint64, C.c_int, C.c_int, _u8p]),
    ("sdb_load_dump_dir", C.c_int, [_ctx, C.c_char_p]),
    ("sdb_nccl_unique_id", C.c_int, [C.c_void_p]),
    ("sdb_broadcast_weights", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int]),
    ("sdb_forward_diffuser", C.c_int, [_ctx, _f32p, C.c_int32, _f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_double, C.c_int,
                                       C.c_int, _f32p, _f32p, _f32p]),
    ("sdb_forward_diffuser_dev", C.c_int, [_ctx, C.c_void_p, C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                           C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("sdb_test_gemm_ex", C.c_int, [_ctx, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                   C.c_int, _f32p]),
    ("sdb_read_dump_tensor", C.c_int64, [C.c_char_p, C.c_int, C.POINTER(C.c_int64), _f32p, C.c_int64]),
    ("sdb_encode_image", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_encode_image_dev", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("sdb_img2img", C.c_int, [_ctx, _u8p, _u8p, _f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_double, C.c_int, C.c_double,
                              _f32p, C.c_uint64, C.c_int, C.c_int, _f32p, _u8p]),
    ("sdb_img2img_dev", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double,
                                  C.c_int, C.c_double, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    ("sdb_sample_ex", C.c_int, [_ctx, _f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, _f32p,
                                _f32p, C.c_uint64, C.c_int, C.c_int, _f32p, _u8p]),
    ("sdb_sample_ex_dev", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int,
                                    C.c_double, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    ("sdb_randn", C.c_int, [_ctx, C.c_uint64, C.c_int64, _f32p]),
    ("sdb_clip_forward", C.c_int, [_ctx, C.POINTER(C.c_int32), C.c_int, C.c_int, _f32p]),
    ("sdb_clip_forward_dev", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("sdb_unet_forward_dev", C.c_int, [_ctx, C.c_void_p, C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p]),
    ("sdb_decode_latent_dev", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("sdb_sample_image_dev", C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_int,
                                       C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("sdb_set_option", C.c_int, [_ctx, C.c_char_p, C.c_int]),
    ("sdb_profile_enable", C.c_int, [_ctx, C.c_int]),
    ("sdb_profile_reset", C.c_int, [_ctx]),
    ("sdb_profile_class_count", C.c_int, [_ctx]),
    ("sdb_profile_get", C.c_int, [_ctx, C.c_int, C.POINTER(C.c_char_p), _i64p, C.POINTER(C.c_double),
                                  C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    ("sdb_profile_get_issued", C.c_int, [_ctx, C.c_int, C.POINTER(C.c_double)]),
    ("sdb_launch_count", C.c_int64, [_ctx]),
    ("sdb_test_linear", C.c_int, [_ctx, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_test_conv2d", C.c_int, [_ctx, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_test_ln_fold", C.c_int, [_ctx, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, _f32p]),
    ("sdb_test_conv_groupnorm", C.c_int, [_ctx, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_int, _f32p, C.POINTER(C.c_int)]),
    ("sdb_test_groupnorm", C.c_int, [_ctx, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p]),
    ("sdb_test_layernorm", C.c_int, [_ctx, _f32p, _f32p, _f32p, C.c_int, C.c_int, _f32p]),
    ("sdb_test_attention", C.c_int, [_ctx, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p]),
]

# sampler ids of sdb_sample_ex (SDB_SAMPLER_* in include/sdb200.h)
SAMPLERS = {"ddim": 0, "dpmpp_2m": 1}

_lib = None


def load():
    """dlopen the in-tree library and type every entry point. Raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, res, args in SIGNATURES:
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def ptr(a: np.ndarray):
    return a.ctypes.data_as(_f32p)


class SdbError(RuntimeError):
    pass


class Context:
    """Owns one sdb_ctx (one CUDA device)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = _ctx()
        rc = self.lib.sdb_create(device, C.byref(h))
        if rc != 0:
            raise SdbError(self.lib.sdb_last_error(None).decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.sdb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise SdbError(self.lib.sdb_last_error(self.h).decode())

    # ---- weights
    def tensor_list(self):
        out = []
        n = self.lib.sdb_tensor_count(self.h)
        for i in range(n):
            name = C.c_char_p()
            dims = (C.c_int64 * 4)()
            nd = C.c_int()
            self.check(self.lib.sdb_tensor_info(self.h, i, C.byref(name), dims, C.byref(nd)))
            out.append((name.value.decode(), tuple(int(dims[j]) for j in range(nd.value))))
        return out

    def set_tensor(self, name, arr):
        a = f32(arr)
        dims = (C.c_int64 * 4)(*a.shape)
        self.check(self.lib.sdb_set_tensor(self.h, name.encode(), ptr(a), dims, a.ndim))

    def get_tensor(self, name, shape):
        a = np.empty(shape, np.float32)
        self.check(self.lib.sdb_get_tensor(self.h, name.encode(), ptr(a), a.size))
        return a

    def init_synthetic(self, seed=0):
        self.check(self.lib.sdb_init_synthetic(self.h, seed))

    def finalize_weights(self):
        self.check(self.lib.sdb_finalize_weights(self.h))

    def weight_arena(self):
        p = C.c_void_p()
        n = C.c_size_t()
        self.check(self.lib.sdb_weight_arena(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def set_option(self, key, value):
        self.check(self.lib.sdb_set_option(self.h, key.encode(), int(value)))

    # ---- hot path (host buffers)
    def unet_forward(self, x, t, context):
        x = f32(x); context = f32(context)
        n, _, H, W = x.shape
        L = context.shape[1]
        out = np.empty_like(x)
        self.check(self.lib.sdb_unet_forward(self.h, ptr(x), int(t), ptr(context), n, H, W, L, ptr(out)))
        return out

    def forward_diffuser(self, latent, t, context, uncond, scale):
        """-> (pred, uncond UNet output, cond UNet output), each [n,4,H,W]."""
        latent = f32(latent); context = f32(context); uncond = f32(uncond)
        n, _, H, W = latent.shape
        outs = [np.empty_like(latent) for _ in range(3)]
        self.check(self.lib.sdb_forward_diffuser(self.h, ptr(latent), int(t), ptr(context), n, context.shape[1], ptr(uncond),
                                                 uncond.shape[0], float(scale), H, W, ptr(outs[0]), ptr(outs[1]), ptr(outs[2])))
        return tuple(outs)

    def nccl_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        if self.lib.sdb_nccl_unique_id(buf) != 0:
            raise SdbError(self.lib.sdb_last_error(None).decode())
        return buf.raw

    def broadcast_weights(self, unique_id: bytes, rank: int, world: int):
        self.check(self.lib.sdb_broadcast_weights(self.h, C.create_string_buffer(unique_id, 128), rank, world))

    def load_dump_dir(self, path):
        self.check(self.lib.sdb_load_dump_dir(self.h, os.fsencode(path)))

    def encode_image(self, img):
        a = f32(img)
        n, ch, H, W = a.shape
        assert ch == 3
        out = np.empty((n, 4, H // 8, W // 8), np.float32)
        self.check(self.lib.sdb_encode_image(self.h, ptr(a), n, H, W, ptr(out)))
        return out

    def clip_forward(self, tokens):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        if t.ndim == 1:
            t = t[None]
        n, L = t.shape
        out = np.empty((n, L, 768), np.float32)
        self.check(self.lib.sdb_clip_forward(self.h, t.ctypes.data_as(C.POINTER(C.c_int32)), n, L, ptr(out)))
        return out

    def decode_latent(self, latent):
        latent = f32(latent)
        n, _, H, W = latent.shape
        img = np.empty((n, 3, 8 * H, 8 * W), np.float32)
        self.check(self.lib.sdb_decode_latent(self.h, ptr(latent), n, H, W, ptr(img)))
        return img

    def sample_latent(self, context, uncond, scale, n_steps, init_latent=None, seed=0, H=64, W=64):
        context = f32(context); uncond = f32(uncond)
        n, L, _ = context.shape
        Lu = uncond.shape[0]
        if init_latent is not None:
            init_latent = f32(init_latent)
            H, W = init_latent.shape[2:]
        out = np.empty((n, 4, H, W), np.float32)
        self.check(self.lib.sdb_sample_latent(self.h, ptr(context), n, L, ptr(uncond), Lu, float(scale), int(n_steps),
                                              ptr(init_latent) if init_latent is not None else None, seed, H, W, ptr(out)))
        return out

    def latent_to_image(self, latent):
        latent = f32(latent)
        n, _, H, W = latent.shape
        rgb = np.empty((n, 8 * H, 8 * W, 3), np.uint8)
        self.check(self.lib.sdb_latent_to_image(self.h, ptr(latent), n, H, W, rgb.ctypes.data_as(_u8p)))
        return rgb

    def sample_image(self, context, uncond, scale, n_steps, init_latent=None, seed=0, H=64, W=64):
        context = f32(context); uncond = f32(uncond)
        n, L, _ = context.shape
        Lu = uncond.shape[0]
        if init_latent is not None:
            init_latent = f32(init_latent)
            H, W = init_latent.shape[2:]
        rgb = np.empty((n, 8 * H, 8 * W, 3), np.uint8)
        self.check(self.lib.sdb_sample_image(self.h, ptr(context), n, L, ptr(uncond), Lu, float(scale), int(n_steps),
                                             ptr(init_latent) if init_latent is not None else None, seed, H, W,
                                             rgb.ctypes.data_as(_u8p)))
        return rgb

    def sample_ex(self, context, uncond, scale, n_steps, sampler="ddim", eta=0.0, init_latent=None, step_noise=None, seed=0,
                  H=64, W=64, latent=True, image=False):
        """Text-to-image with a selectable sampler (sdb_sample_ex): sampler "ddim" (eta in [0,1]) or "dpmpp_2m" (eta 0).
        step_noise [T,n,4,H,W] (DDIM with eta > 0) or None (the seeded stream). -> (latent [n,4,H,W] or None, rgb
        [n,8H,8W,3] u8 or None); `latent` / `image` select the outputs."""
        context = f32(context); uncond = f32(uncond)
        n, L, _ = context.shape
        if isinstance(sampler, str) and sampler not in SAMPLERS:
            raise ValueError(f"sampler must be one of {sorted(SAMPLERS)}, got {sampler!r}")
        sid = SAMPLERS[sampler] if isinstance(sampler, str) else int(sampler)  # an int id goes to the library as is
        if init_latent is not None:
            init_latent = f32(init_latent)
            H, W = init_latent.shape[2:]
        if step_noise is not None:
            step_noise = f32(step_noise)
            T = len(range(999, -1, -(1000 // int(n_steps)))) if 1 <= int(n_steps) <= 1000 else 0
            if step_noise.shape != (T, n, 4, H, W):
                raise ValueError(f"step_noise must be [T, n, 4, H, W] = {(T, n, 4, H, W)}, got {step_noise.shape}")
        lat = np.empty((n, 4, H, W), np.float32) if latent else None
        rgb = np.empty((n, 8 * H, 8 * W, 3), np.uint8) if image else None
        opt = lambda a: ptr(a) if a is not None else None
        self.check(self.lib.sdb_sample_ex(self.h, ptr(context), n, L, ptr(uncond), uncond.shape[0], float(scale), int(n_steps),
                                          sid, float(eta), opt(init_latent), opt(step_noise), int(seed), H, W,
                                          opt(lat), rgb.ctypes.data_as(_u8p) if rgb is not None else None))
        return lat, rgb

    def randn(self, seed, count):
        """The library's seeded N(0,1) stream (sdb_randn): `count` float32 values."""
        out = np.empty(int(count), np.float32)
        self.check(self.lib.sdb_randn(self.h, int(seed), int(count), ptr(out)))
        return out

    def img2img(self, context, uncond, scale, n_steps, rgb, strength, mask=None, noise=None, seed=0, latent=True, image=True):
        """rgb [n,8H,8W,3] u8, mask [n,8H,8W] (nonzero = repaint) or None, noise [n,4,H,W] or None (seeded stream).
        -> (latent [n,4,H,W] or None, rgb [n,8H,8W,3] u8 or None); `latent` / `image` select the outputs."""
        context = f32(context); uncond = f32(uncond)
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        n, L, _ = context.shape
        if rgb.ndim != 4 or rgb.shape[0] != n or rgb.shape[3] != 3:
            raise ValueError(f"rgb must be [n={n}, 8H, 8W, 3] uint8, got {rgb.shape}")
        H, W = rgb.shape[1] // 8, rgb.shape[2] // 8
        if rgb.shape[1] != 8 * H or rgb.shape[2] != 8 * W:
            raise ValueError(f"image height and width must be multiples of 8, got {rgb.shape[1:3]}")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
            if mask.shape != rgb.shape[:3]:
                raise ValueError(f"mask must be [n, 8H, 8W] = {rgb.shape[:3]}, got {mask.shape}")
        if noise is not None:
            noise = f32(noise)
            if noise.shape != (n, 4, H, W):
                raise ValueError(f"noise must be [n, 4, H, W] = {(n, 4, H, W)}, got {noise.shape}")
        lat = np.empty((n, 4, H, W), np.float32) if latent else None
        out = np.empty_like(rgb) if image else None
        self.check(self.lib.sdb_img2img(self.h, rgb.ctypes.data_as(_u8p), mask.ctypes.data_as(_u8p) if mask is not None else None,
                                        ptr(context), n, L, ptr(uncond), uncond.shape[0], float(scale), int(n_steps),
                                        float(strength), ptr(noise) if noise is not None else None, int(seed), H, W,
                                        ptr(lat) if lat is not None else None, out.ctypes.data_as(_u8p) if out is not None else None))
        return lat, out

    # ---- profiling
    def profile(self, on=True):
        self.check(self.lib.sdb_profile_enable(self.h, 1 if on else 0))

    def profile_reset(self):
        self.check(self.lib.sdb_profile_reset(self.h))

    def profile_table(self):
        rows = {}
        for i in range(self.lib.sdb_profile_class_count(self.h)):
            name = C.c_char_p(); ln = C.c_int64(); ms = C.c_double(); fl = C.c_double(); by = C.c_double()
            self.check(self.lib.sdb_profile_get(self.h, i, C.byref(name), C.byref(ln), C.byref(ms), C.byref(fl), C.byref(by)))
            iss = C.c_double()
            self.check(self.lib.sdb_profile_get_issued(self.h, i, C.byref(iss)))
            rows[name.value.decode()] = dict(launches=ln.value, ms=ms.value, flops=fl.value, bytes=by.value, issued_flops=iss.value)
        return rows

    def launch_count(self):
        return int(self.lib.sdb_launch_count(self.h))

    # ---- single-kernel test entries
    def test_linear(self, a, w, bias=None, passes=1):
        a = f32(a); w = f32(w)
        M, K = a.shape; N = w.shape[1]
        out = np.empty((M, N), np.float32)
        b = f32(bias) if bias is not None else None
        self.check(self.lib.sdb_test_linear(self.h, ptr(a), ptr(w), ptr(b) if b is not None else None, M, K, N, passes, ptr(out)))
        return out

    def test_gemm_ex(self, a, w, bias=None, residual=None, passes=1, geglu=False, from_f16=False, xa=None, xw=None):
        a = f32(a); w = f32(w)
        M, K = a.shape; N = w.shape[1]
        out = np.empty((M, N // 2 if geglu else N), np.float32)
        opt = lambda v: (None, None) if v is None else (f32(v), ptr(f32(v)))
        keep = [opt(bias), opt(residual), opt(xa), opt(xw)]
        for i, (arr, _) in enumerate(keep):  # keep the contiguous copies alive across the call
            if arr is not None:
                keep[i] = (arr, ptr(arr))
        XK = 0 if xa is None else keep[2][0].shape[1]
        self.check(self.lib.sdb_test_gemm_ex(self.h, ptr(a), ptr(w), keep[0][1], keep[1][1], M, K, N, passes,
                                             (1 if geglu else 0) | (4 if from_f16 else 0), keep[2][1], keep[3][1], XK, ptr(out)))
        return out

    def test_conv2d(self, x, w, bias=None, stride=1, upsample=0, passes=1):
        x = f32(x); w = f32(w)
        n, cin, H, W = x.shape
        cout, _, k, _ = w.shape
        Ho = 2 * H if upsample else (H // 2 if stride == 2 else H)
        Wo = 2 * W if upsample else (W // 2 if stride == 2 else W)
        y = np.empty((n, cout, Ho, Wo), np.float32)
        b = f32(bias) if bias is not None else None
        self.check(self.lib.sdb_test_conv2d(self.h, ptr(x), ptr(w), ptr(b) if b is not None else None, n, cin, H, W, cout,
                                            k, stride, upsample, passes, ptr(y)))
        return y

    def test_ln_fold(self, a, w0, b0, gamma, beta, w1, b1=None, a2=None, passes=3, geglu=False):
        a, w0, b0, gamma, beta, w1 = (f32(v) for v in (a, w0, b0, gamma, beta, w1))
        b1 = f32(b1) if b1 is not None else None
        a2 = f32(a2) if a2 is not None else None
        M, K0 = a.shape; Cc = w0.shape[1]; N = w1.shape[1]
        out = np.empty((M, N // 2 if geglu else N), np.float32)
        self.check(self.lib.sdb_test_ln_fold(self.h, ptr(a), ptr(a2) if a2 is not None else None, ptr(w0), ptr(b0), ptr(gamma),
                                             ptr(beta), ptr(w1), ptr(b1) if b1 is not None else None, M, K0, Cc, N, passes,
                                             1 if geglu else 0, ptr(out)))
        return out

    def test_conv_groupnorm(self, x, w, bias, gamma, beta, passes=3, silu=False):
        x = f32(x); w = f32(w); bias = f32(bias); gamma = f32(gamma); beta = f32(beta)
        n, cin, H, W = x.shape
        cout, _, k, _ = w.shape
        y = np.empty((n, cout, H, W), np.float32)
        slots = C.c_int()
        self.check(self.lib.sdb_test_conv_groupnorm(self.h, ptr(x), ptr(w), ptr(bias), ptr(gamma), ptr(beta), n, cin, H, W, cout, k,
                                                    passes, 1 if silu else 0, ptr(y), C.byref(slots)))
        return y, slots.value

    def test_groupnorm(self, x, gamma, beta, silu=False):
        x = f32(x); n, c, H, W = x.shape
        y = np.empty_like(x)
        g = f32(gamma); b = f32(beta)
        self.check(self.lib.sdb_test_groupnorm(self.h, ptr(x), ptr(g), ptr(b), n, c, H, W, 1 if silu else 0, ptr(y)))
        return y

    def test_layernorm(self, x, gamma, beta):
        x = f32(x); rows, c = x.shape
        y = np.empty_like(x)
        g = f32(gamma); b = f32(beta)
        self.check(self.lib.sdb_test_layernorm(self.h, ptr(x), ptr(g), ptr(b), rows, c, ptr(y)))
        return y

    def test_attention(self, q, k, v, heads):
        q = f32(q); k = f32(k); v = f32(v)
        n, Nq, Cc = q.shape; Nk = k.shape[1]
        out = np.empty_like(q)
        self.check(self.lib.sdb_test_attention(self.h, ptr(q), ptr(k), ptr(v), n, Nq, Nk, Cc, heads, ptr(out)))
        return out
