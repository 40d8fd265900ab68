"""Shared fixtures for the -m gpu parity tests: seeded parameters, normalisation, inputs, device views, the names of
the kernels a call launches, the oracle of whole batches with the parity bars of the tensor path, and the rmbe
post-filter's weights and oracle."""
import collections
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


def kernel_counts(codec, fn):
    """How often each kernel is launched by one call fn(), by name without the parameter list ('fused_enc_kernel',
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
    return collections.Counter(names)


def kernels_of(codec, fn):
    """The names of the kernels one call fn() launches (kernel_counts without the counts)."""
    return set(kernel_counts(codec, fn))


def ran(names, kernel):
    """kernel ('fused_enc_kernel', or with template arguments: 'f16_first_s2_tma_kernel<true>') is among names."""
    return kernel in names or kernel in {n.split("<")[0] for n in names}


def fmt(names):
    return ", ".join(sorted(names))


# ---- oracle references of whole batches and the parity bars of the tensor path -------------------------------------
ORACLE_BATCH = 192  # patches per oracle call: one 2048x1536 image at P = 128 (a whole batch of them would need GBs)


def crops(images, P):
    return np.stack([p for im in images for p in O.crop_image_input_patches(im, P)])


def oracle_encoder(patches, variant, enc, mean=MEAN, std=STD, q=2):
    return np.concatenate([O.encoder(patches[i:i + ORACLE_BATCH].astype(np.float32), variant, enc, mean, std, q)
                           for i in range(0, len(patches), ORACLE_BATCH)])


def oracle_decoder(symbols, variant, dec, mean=MEAN, std=STD, q=2):
    return np.concatenate([O.decoder(symbols[i:i + ORACLE_BATCH], variant, dec, mean, std, q)
                           for i in range(0, len(symbols), ORACLE_BATCH)])


def logits64(patches, variant, enc, mean, std):
    return np.concatenate([O.encoder_logits(patches[i:i + ORACLE_BATCH].astype(np.float32), variant, enc, mean, std,
                                            dtype=torch.float64) for i in range(0, len(patches), ORACLE_BATCH)])


def check_symbols(got, ref, patches, variant, enc, mean=MEAN, std=STD):
    """q = 2: at most 1e-5 of the symbols (or one) differ from the oracle, and each difference sits where the fp64 logit
    is within fp32 noise of 0 (test_gpu_parity.py's rule).  fp64 logits are evaluated for the patches with a mismatch only.
    Returns (mismatches, largest |fp64 logit| at a mismatch)."""
    got = np.asarray(got).reshape(ref.shape)
    diff = got != ref
    nm = int(diff.sum())
    assert nm <= max(1, 1e-5 * ref.size), f"{nm}/{ref.size} symbol mismatches"
    if not nm:
        return 0, 0.0
    bad = np.flatnonzero(diff.reshape(len(ref), -1).any(1))
    l64 = logits64(patches[bad], variant, enc, mean, std)
    at = np.abs(l64[diff[bad]])
    bound = 1.5e-7 + 4e-6 * np.abs(l64).max()
    assert at.max() < bound, f"mismatch at |fp64 logit| {at.max():.3e} outside the dead zone (< {bound:.3e})"
    return nm, float(at.max())


def check_recon(rec_f, rec_u8, want_f):
    """float32 within 1e-3 max-abs of the oracle, uint8 within one grey level of np.around of it at a rate < 1e-4.
    Returns (max-abs float error, fraction of u8 values that differ)."""
    err = float(np.abs(np.asarray(rec_f) - want_f).max())
    assert err <= 1e-3, f"reconstruction max-abs error {err:.3e}"
    d = np.abs(np.asarray(rec_u8).astype(np.int32) - O.around_u8(want_f).astype(np.int32))
    assert d.max() <= 1 and (d != 0).mean() < 1e-4, (int(d.max()), float((d != 0).mean()))
    return err, float((d != 0).mean())


def oracle_images(symbols, H, W, P, variant, dec, mean=MEAN, std=STD):
    """The oracle decoder of [B, gh*gw, ...] symbols, stitched and cropped like utils.concat_patches: [B,H,W,3] f32."""
    return np.stack([O.concat_patches(list(oracle_decoder(s, variant, dec, mean, std)), H, W, P) for s in symbols])


# ---- the rmbe post-filter: fan-in weights, their normalisation and the fp32 oracle on whole images --------------------
PM = np.array([110.0, 108.0, 99.0], np.float32)  # post-filter normalisation of the fan-in weight set
PS = np.array([55.0, 57.0, 60.0], np.float32)
ORACLE_TILES = 64  # tiles per oracle call (a 2048x1536 pass at once would need GBs of activations)


def post_params(name="rmbe"):
    """Fan-in weights: far from the identity, so a tile read before or after the other pass's write shows."""
    return O.init_params(O.POSTFILTERS[name], 3, 77 if name == "rmbe" else 78, "fanin")


def in_tiles(run, tiles):
    return np.concatenate([run(tiles[i:i + ORACLE_TILES]) for i in range(0, len(tiles), ORACLE_TILES)])


def oracle32(img, name, pp, mean=PM, std=PS):
    return O.rmbe(img, lambda t: in_tiles(lambda x: O.postfilter(x, name, pp, mean, std), t))
