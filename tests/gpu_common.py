"""Shared fixtures for the -m gpu parity tests: seeded parameters, normalisation, inputs, device views and the names of
the kernels a call launches."""
import json
import os
import tempfile

import numpy as np
import torch

from oracle import codec_oracle as O
import tf_image_compression_b200 as T

MEAN = np.array([118.3, 113.9, 102.6], np.float32)
STD = np.array([61.7, 59.2, 63.8], np.float32)


def params_for(variant, scheme, seed=1234, q=2):
    ov = O.VARIANTS[variant]
    enc = O.init_params(ov["enc"], 3, seed, scheme)
    dec = O.init_params(ov["dec"], ov["bottleneck"], seed + 1, scheme)
    if scheme == "fanin":
        dec = O.condition_decoder(variant, dec, q)
    return enc, dec


def make_codec(variant, scheme="fanin", q=2, compute="fp32", seed=1234):
    enc, dec = params_for(variant, scheme, seed, q)
    c = T.Codec(variant, quan_scale=q, mean=MEAN, std=STD, enc_params=enc, dec_params=dec, compute=compute)
    return c, enc, dec


def patches_from_images(n_images, h, w, P, seed=0, kind="natural"):
    out = []
    for i in range(n_images):
        out += O.crop_image_input_patches(O.synthetic_image(h, w, seed + i, kind), P)
    return np.stack(out)


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def seeded_u8(shape, seed):
    """Uniform u8 noise from a seeded torch generator, as bench.py makes its images."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).numpy()


def device_view(host, offset, dtype=torch.uint8):
    """host's values on the device, at byte `offset` from a 512-byte aligned allocation."""
    t = torch.from_numpy(np.ascontiguousarray(host))
    esz = t.element_size()
    assert offset % esz == 0
    buf = torch.zeros(t.numel() + 64 // esz, dtype=dtype, device="cuda")
    v = buf[offset // esz:offset // esz + t.numel()].view(tuple(t.shape))
    v.copy_(t.to("cuda"))
    assert v.data_ptr() % 512 == offset and v.is_contiguous()
    return v


def _short(name):
    name = name.replace("(anonymous namespace)::", "").removeprefix("void ")
    return name.split("(")[0].rsplit("::", 1)[-1].strip()


def kernels_of(codec, fn):
    """The names of the kernels one call fn() launches, without their parameter lists ('fused_enc_kernel',
    'f16_first_s2_tma_kernel<true>', ...), from torch.profiler with CUDA activities.  fn() runs once before, so that
    lazily built weight images are not counted; a torch kernel opens the profiled window, and the kernels recorded must
    be as many as the codec counts (codec.launch_count), so that a kernel the profiler missed cannot pass for a path
    that was not taken."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device="cuda").add_(1)
        n0 = codec.launch_count
        fn()
        torch.cuda.synchronize()
        launched = codec.launch_count - n0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    names = [_short(e["name"]) for e in events if e.get("cat") == "kernel" and "at::native" not in e["name"]]
    assert len(names) == launched, f"torch.profiler recorded {len(names)} kernels, the codec launched {launched}: {names}"
    return set(names)


def ran(names, kernel):
    """kernel ('fused_enc_kernel', or with template arguments: 'f16_first_s2_tma_kernel<true>') is among names."""
    return kernel in names or kernel in {n.split("<")[0] for n in names}


def fmt(names):
    return ", ".join(sorted(names))
