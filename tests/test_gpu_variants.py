"""-m gpu parity of the codecs the reference submitted, on whole images: model_3 (submit/2, submit/3, base_model/fin) and
model_2 (submit/1), both at P = 128.  In tensor mode they run code model_0 never reaches: a stride-2 quantiser (8
epilogue warps instead of 16), 80 bottleneck channels (model_3), a CUDA-core decode_4 inside the tensor-mode graph that
reads the symbols through the inverse-sigmoid table (model_3: u16_supported rejects cin = 80), a 64 -> 64 transposed
conv fed from symbols by u16_split_symlut_kernel (model_2), the stand-alone 32 -> 3 image-writing transposed conv
(decode_2 is 64 -> 32, so the fused decoder pair does not apply), no fused encoder (encode_2 is 32 -> 64) and residual
blocks at 32x32x64 on both sides of model_3.

Bars as in test_gpu_scale_parity.py (gpu_common.check_symbols / check_recon): symbol mismatch rate <= 1e-5 (or one) and
each mismatch in the fp64 dead zone; reconstruction within 1e-3 max-abs as float32, within one grey level at a rate
< 1e-4 as uint8; the histogram equal to np.bincount of the returned symbols.  The submit/2 flow adds the post-filter
bars of test_gpu_postfilter.py.  Every case prints its errors and, in tensor mode, the kernels that ran."""
import os
import time

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
from tf_image_compression_b200 import entry, range_coder
from gpu_common import (PM, PS, check_recon, check_symbols, crops, device_view, fmt, kernel_counts, kernels_of,
                        make_codec, oracle32, oracle_encoder, oracle_images, params_for, post_params, ran, seeded_u8)

pytestmark = pytest.mark.gpu

VARIANTS = ["model_3", "model_2"]
MODES = ["tensor", "fp32"]
P = 128

_cache = {}


def cached(key, fn):
    """Oracle results are shared by the compute modes, offsets and chunk sizes that check against them."""
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def reference(variant, H, W, B):
    """Seeded u8 images [B,H,W,3], their patches, the oracle's symbols [B, gh*gw, hb, wb, cb] and the oracle decoder's
    stitched images of those symbols [B,H,W,3] f32."""
    def run():
        enc, dec = params_for(variant, "fanin")
        imgs = seeded_u8((B, H, W, 3), 100 + H + W)
        patches = crops(imgs, P)
        ref = oracle_encoder(patches, variant, enc)
        ref = ref.reshape(B, -1, *ref.shape[1:])
        return imgs, patches, ref, oracle_images(ref, H, W, P, variant, dec)
    return cached((variant, H, W, B), run)


def no_tensor_kernels(names):
    return not any(n.startswith(("f16_", "u16", "umma", "fused")) for n in names)


# ---- 1. image-level dispatch matrix -------------------------------------------------------------------------------------
# (id, images H x W x count, byte offset of the device input)
DISPATCH_CASES = [
    ("exact0", (512, 768, 4), 0),
    ("exact1", (512, 768, 4), 1),
    ("exact4", (512, 768, 4), 4),
    # reflect-padded images; the 2- and 3-pixel sides reflect over many periods
    ("ragged2x130", (2, 130, 3), 0),
    ("ragged129x385", (129, 385, 2), 0),
    ("ragged1356x2040", (1356, 2040, 1), 0),
]


def check_dispatch(variant, exact_aligned, k_enc, k_dec):
    """Tensor mode: the first layer reads u8 images through TMA only on an aligned exact grid, else through the gather
    kernel; neither fused pair applies; the u16 trunk runs.  model_3's decode_4 (cin = 80) is the CUDA-core transposed
    conv reading symbols; model_2's is a u16 deconv fed by the symbol -> pair-plane split."""
    if exact_aligned:
        assert ran(k_enc, "f16_first_s2_tma_kernel<false>") and not ran(k_enc, "f16_first_s2_kernel"), fmt(k_enc)
    else:
        assert ran(k_enc, "f16_first_s2_kernel") and not ran(k_enc, "f16_first_s2_tma_kernel"), fmt(k_enc)
    assert not ran(k_enc, "fused_enc_kernel") and not any(n.endswith("_simt_kernel") for n in k_enc), fmt(k_enc)
    assert not ran(k_dec, "fused_dec_kernel") and ran(k_dec, "u16_pair_kernel"), fmt(k_dec)
    if variant == "model_3":
        assert ran(k_dec, "deconv3x3_simt_kernel") and not ran(k_dec, "u16_split_symlut_kernel"), fmt(k_dec)
    else:
        assert ran(k_dec, "u16_split_symlut_kernel") and not any(n.endswith("_simt_kernel") for n in k_dec), fmt(k_dec)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", DISPATCH_CASES, ids=[c[0] for c in DISPATCH_CASES])
@pytest.mark.parametrize("variant", VARIANTS)
def test_image_dispatch_against_oracle(variant, case, mode):
    """encode_images of u8 device images against the oracle (crop with np.pad 'reflect', encode), with the histogram;
    decode_images of the oracle's symbols, float32 and u8, against the oracle decoder stitched and cropped.  A misaligned
    input must give the aligned call's symbols (up to the dead zone), and a decode into a misaligned output the same
    bytes as the aligned decode."""
    t0 = time.perf_counter()
    name, (H, W, B), off = case
    codec, enc, dec = make_codec(variant, compute=mode)
    imgs, patches, ref, want = reference(variant, H, W, B)
    d_imgs = device_view(imgs, off)
    codec.hist_reset()
    sym = codec.encode_images(d_imgs, P)
    counts = codec.hist_read()
    sym_h = sym.cpu().numpy()
    assert sym_h.shape == ref.shape, (sym_h.shape, ref.shape)
    assert np.array_equal(counts, np.bincount(sym_h.reshape(-1), minlength=2).astype(np.uint64))
    nm, worst = check_symbols(sym_h, ref.reshape(-1, *ref.shape[2:]), patches, variant, enc)
    d_ref = torch.from_numpy(ref).cuda()
    rec_f = codec.decode_images(d_ref, H, W, P, out_dtype=np.float32)
    rec_u8 = codec.decode_images(d_ref, H, W, P)
    codec.check_status()
    err, rate8 = check_recon(rec_f.cpu().numpy(), rec_u8.cpu().numpy(), want)
    k_enc = kernels_of(codec, lambda: codec.encode_images(d_imgs, P))
    k_dec = kernels_of(codec, lambda: codec.decode_images(d_ref, H, W, P, out_dtype=np.float32))
    k_dec8 = kernels_of(codec, lambda: codec.decode_images(d_ref, H, W, P))
    if mode == "tensor":
        check_dispatch(variant, name == "exact0", k_enc, k_dec)
        check_dispatch(variant, name == "exact0", k_enc, k_dec8)
    else:
        assert no_tensor_kernels(k_enc | k_dec | k_dec8), fmt(k_enc | k_dec | k_dec8)
    if off:
        aligned = codec.encode_images(device_view(imgs, 0), P).cpu().numpy()
        check_symbols(sym_h, aligned.reshape(-1, *ref.shape[2:]), patches, variant, enc)
        out8 = device_view(np.zeros((B, H, W, 3), np.uint8), off)
        codec.decode_images(d_ref, H, W, P, out=out8)
        assert torch.equal(out8, rec_u8)
        if off % 4 == 0:
            outf = device_view(np.zeros((B, H, W, 3), np.float32), off, torch.float32)
            codec.decode_images(d_ref, H, W, P, out=outf)
            assert torch.equal(outf, rec_f)
    print(f"[1 {variant} {name} {mode}] {B} x {H}x{W}, {len(patches)} patches, {ref.size} symbols; mismatches {nm} "
          f"(max |fp64 logit| {worst:.2e}); recon max-abs {err:.2e}, u8 differing {rate8:.1e}; encode: {fmt(k_enc)}; "
          f"decode: {fmt(k_dec)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- 2. launch counts ----------------------------------------------------------------------------------------------------
# Launches per call on 4 exact-grid 256x384 images (24 patches: under the 64 patches from which run_graph splits a graph
# into L2-sized groups, so every layer runs once over all patches).  Derived from run_graph / launch_u16 and confirmed on
# a B200; a layer that silently changes plan (slices, a fallback kernel, a conversion launch) changes the count.
# model_3 encoder, 14:  encode_1 (3 -> 32, TMA first layer) 1 + encode_2 (32 -> 64, stride 2) 1 + encode_res_m1/0 at
#   32x32x64 4 + encode_3 (stride 2, 32-channel K-blocks) 1 + encode_res_1/2/3 at 16x16x64 6 + encode_4 (64 -> 80,
#   stride 2, quantiser epilogue) 1: all 80 output channels in one launch.
# model_3 decoder, 15:  decode_4 (80 -> 64 on the CUDA cores, reads the symbols; no split launch because layer 0 is not
#   u16-capable) 1 + decode_res_1/2/3 at 16x16 6 + decode_3 (64 -> 64 transposed: two phase-stacked 32-channel slices) 2
#   + decode_res_4/5 at 32x32 4 + decode_2 (64 -> 32) 1 + decode_1 (32 -> 3 into the image) 1.
# model_2 encoder, 8:  encode_1 1 + encode_2 1 + encode_3 1 + encode_res_1/2 4 + encode_4 (64 -> 64, stride 2) 1.
# model_2 decoder, 11:  symbols -> pair planes (u16_split_symlut_kernel) 1 + decode_4 (64 -> 64 transposed) 2 slices +
#   decode_res_1/2 4 + decode_3 2 slices + decode_2 1 + decode_1 1.
LAUNCHES = {"model_3": (14, 15), "model_2": (8, 11)}


@pytest.mark.parametrize("variant", VARIANTS)
def test_launch_counts(variant):
    """Launches per encode_images / decode_images call in tensor mode (LAUNCHES, with the derivation), counted by the
    codec, and the kernels the profiler saw per name."""
    codec, _, _ = make_codec(variant, compute="tensor")
    imgs = torch.from_numpy(np.stack([O.synthetic_image(256, 384, 80 + i) for i in range(4)])).cuda()
    sym = codec.encode_images(imgs, P)  # first calls: lazily built weight images add launches
    codec.decode_images(sym, 256, 384, P)
    c_enc = kernel_counts(codec, lambda: codec.encode_images(imgs, P))
    c_dec = kernel_counts(codec, lambda: codec.decode_images(sym, 256, 384, P))
    n0 = codec.launch_count
    codec.encode_images(imgs, P)
    n1 = codec.launch_count
    codec.decode_images(sym, 256, 384, P)
    n2 = codec.launch_count
    print(f"[2 {variant}] encode {n1 - n0} launches: {dict(sorted(c_enc.items()))}; decode {n2 - n1} launches: "
          f"{dict(sorted(c_dec.items()))}")
    assert (n1 - n0, n2 - n1) == LAUNCHES[variant], (n1 - n0, n2 - n1)
    assert (sum(c_enc.values()), sum(c_dec.values())) == LAUNCHES[variant]
    codec.close()


# ---- 3. chunk boundaries -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [1, 7, 25, 4096])
@pytest.mark.parametrize("variant", VARIANTS)
def test_chunk_boundaries(variant, chunk):
    """set_chunk_patches(c) in tensor mode with host and device buffers, on the 4 x 512x768 images of the dispatch matrix
    (24 patches each): image calls run whole images per chunk (at least one), patch calls cut the images anywhere.
    encode / decode (u8 and f32) / round trip results are bit-identical to the one-chunk call, whose symbols and
    reconstruction match the oracle.  For model_3, c = 1 and 7 put the CUDA-core symbol reader's patch offset (geo.n0)
    on every chunk."""
    t0 = time.perf_counter()
    B, H, W = 4, 512, 768
    codec, enc, dec = make_codec(variant, compute="tensor")
    imgs, patches, ref, want = reference(variant, H, W, B)
    sym = codec.encode_images(imgs, P)
    rec_u8 = codec.decode_images(sym, H, W, P)
    rec_f = codec.decode_images(sym, H, W, P, out_dtype=np.float32)
    nm, worst = check_symbols(sym, ref.reshape(-1, *ref.shape[2:]), patches, variant, enc)
    if nm == 0:  # the reconstruction of the oracle's symbols
        check_recon(rec_f, rec_u8, want)
    psym = sym.reshape(-1, *sym.shape[2:])
    prec = codec.decode_patches(psym)
    codec.set_chunk_patches(chunk)
    for dev in (False, True):
        put = (lambda a: torch.from_numpy(a).cuda()) if dev else (lambda a: a)
        get = (lambda t: t.cpu().numpy()) if dev else (lambda a: a)
        assert np.array_equal(get(codec.encode_images(put(imgs), P)), sym), dev
        assert np.array_equal(get(codec.decode_images(put(sym), H, W, P)), rec_u8), dev
        assert np.array_equal(get(codec.decode_images(put(sym), H, W, P, out_dtype=np.float32)), rec_f), dev
        r, s = codec.roundtrip_images(put(imgs), P)
        assert np.array_equal(get(s), sym) and np.array_equal(get(r), rec_u8), dev
        assert np.array_equal(get(codec.encode_patches(put(patches))), psym), dev
        assert np.array_equal(get(codec.decode_patches(put(psym))), prec), dev
    codec.check_status()
    print(f"[3 {variant} chunk {chunk}] {len(patches)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); host and "
          f"device bit-identical to one chunk; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- 4. submit/2 end to end ----------------------------------------------------------------------------------------------
def test_submit2_compress_uncompress_postfilter(tmp_path):
    """submit/2: model_3 in tensor mode with the rmbe post-filter (fan-in weights of test_gpu_postfilter.py).
    entry.compress(coder='gpu') of 1536x2048, 512x768 twice and 500x700 (ragged, and not a multiple of the rmbe tile),
    then entry.uncompress(postfilter=True) with the gpu, host and serial coders.  The three are identical and equal
    round_u8(postfilter_images(decode_images(..., float32))) composed by hand, bitwise.  Against the oracle:
    - the decoded float within check_recon of the oracle decoder;
    - postfilter_images of the decoded float within 2e-3 of oracle32 of the same input;
    - the whole float chain within 3e-3 of O.decoder -> O.concat_patches -> O.rmbe (the post-filter's bar where the
      decoder runs first);
    - the u8 output at most one grey level from np.around of the oracle chain, and only where the oracle's float is
      within 3e-3 of a .5 boundary."""
    t0 = time.perf_counter()
    codec, _, dec = make_codec("model_3", compute="tensor")
    pp = post_params()
    codec.set_postfilter(pp, PM, PS)
    shapes = [(1536, 2048), (512, 768), (500, 700), (512, 768)]
    images = [O.synthetic_image(h, w, 90 + i) for i, (h, w) in enumerate(shapes)]
    names = [f"img_{i}" for i in range(len(images))]
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=P)
    codec.hist_reset()
    for im in images:
        codec.encode_images(im[None], P)
    counts = codec.hist_read().astype(np.float64)
    prob = counts / counts.sum()
    cum = entry.cum_freq_table(prob, cfg["resolution"])
    files = entry.compress(codec, images, names, cfg, prob, str(tmp_path / "enc"), coder="gpu")
    outs = {c: entry.uncompress(codec, str(tmp_path / "enc"), cfg, prob, postfilter=True, coder=c)
            for c in ("gpu", "host", "serial")}
    codec.check_status()
    for c in ("host", "serial"):
        assert sorted(outs[c]) == sorted(outs["gpu"]) == sorted(names)
        assert all(np.array_equal(outs[c][n], outs["gpu"][n]) for n in names), c
    e_dec = e_pf = e_chain = 0.0
    n8 = 0
    for (path, _), name, im in zip(files, names, images):
        H, W, _ = im.shape
        stem, eshape, n, h, w = entry.parse_encoded_name(os.path.basename(path), cfg)
        assert (stem, h, w) == (name, H, W)
        with open(path, "rb") as f:
            seq = range_coder.decode_streams([f.read()], [n], cum)[0]
        sym = np.asarray(seq, np.uint8).reshape(1, -1, *eshape)
        d_sym = torch.from_numpy(sym).cuda()
        img = codec.decode_images(d_sym, H, W, P, out_dtype=np.float32)
        dec_gpu = img.cpu().numpy()[0]
        codec.postfilter_images(img)
        out8 = codec.round_u8(img).cpu().numpy()[0]
        got = img.cpu().numpy()[0]
        codec.check_status()
        assert np.array_equal(out8, outs["gpu"][name]), f"{name}: uncompress != the hand composition"
        want_dec = oracle_images(sym, H, W, P, "model_3", dec)[0]
        e, _ = check_recon(dec_gpu, codec.decode_images(d_sym, H, W, P).cpu().numpy()[0], want_dec)
        e_dec = max(e_dec, e)
        ep = float(np.abs(got - oracle32(dec_gpu, "rmbe", pp)).max())
        want = oracle32(want_dec, "rmbe", pp)
        ec = float(np.abs(got - want).max())
        d = np.abs(out8.astype(np.int32) - O.around_u8(want).astype(np.int32))
        near = np.abs(want - np.floor(want) - 0.5) <= 3e-3
        print(f"  [4 {name} {H}x{W}] decode |gpu-oracle32| {e:.3e}; rmbe of the gpu decode |gpu-oracle32| {ep:.3e}; "
              f"chain |gpu-oracle32| {ec:.3e}; u8 differing {int((d != 0).sum())}")
        assert ep <= 2e-3, (name, ep)
        assert ec <= 3e-3, (name, ec)
        assert d.max() <= 1 and not (d[~near] != 0).any(), f"{name}: u8 differs away from a .5 boundary"
        e_pf, e_chain, n8 = max(e_pf, ep), max(e_chain, ec), n8 + int((d != 0).sum())
    print(f"[4 submit/2] {len(images)} images; decode {e_dec:.2e}, rmbe {e_pf:.2e}, chain {e_chain:.2e}; u8 differing "
          f"{n8}; gpu / host / serial identical; {time.perf_counter() - t0:.1f} s")
    codec.close()
