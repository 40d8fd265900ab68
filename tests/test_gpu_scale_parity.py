"""-m gpu parity of the tensor-core path (compute = tensor) against the CPU oracle where the small fixtures do not reach:
the benchmark workload element by element, patch counts around the waves of the persistent CTA-pair kernels, chunk
boundaries, every first-layer / fused-pair dispatch path (checked by the names of the kernels that ran) and
quan_scale > 2.  Tolerances as in test_gpu_parity.py: symbol mismatch rate <= 1e-5 and every mismatch where the fp64
logit is within fp32 noise of the sigmoid == 0.5 threshold; reconstruction within 1e-3 max-abs as float32, within one
grey level at a rate < 1e-4 as uint8."""
import time

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
from gpu_common import (MEAN, STD, check_recon, check_symbols, crops, device_view, fmt, kernels_of, logits64, make_codec,
                        oracle_decoder, oracle_encoder, oracle_images, params_for, ran, seeded_u8)
import tf_image_compression_b200 as T

pytestmark = pytest.mark.gpu

# ---- A. the benchmark workload --------------------------------------------------------------------------------------
def test_benchmark_workload_against_oracle():
    """BASELINE config 2 as bench.py times it: model_0, compute = tensor, 64 x 2048x1536 u8 images resident on the device,
    P = 128, default chunking (12 288 patches, 50.3 M symbols).  Every symbol against the oracle, the histogram against
    np.bincount, decode_images of the GPU's symbols (float32 and u8) against the oracle decoder on every pixel, and the
    streamed host-buffer round trip bit-identical to the device-resident calls."""
    t0 = time.perf_counter()
    B, H, W, P = 64, 1536, 2048, 128
    codec, enc, dec = make_codec("model_0", compute="tensor")
    imgs = seeded_u8((B, H, W, 3), 1234)
    d_imgs = torch.from_numpy(imgs).cuda()
    codec.hist_reset()
    sym = codec.encode_images(d_imgs, P)
    counts = codec.hist_read()
    rec_u8 = codec.decode_images(sym, H, W, P)
    k_enc = kernels_of(codec, lambda: codec.encode_images(d_imgs, P))
    k_dec = kernels_of(codec, lambda: codec.decode_images(sym, H, W, P))
    rec_f = codec.decode_images(sym, H, W, P, out_dtype=np.float32)
    sym_h = sym.cpu().numpy()
    assert np.array_equal(counts, np.bincount(sym_h.reshape(-1), minlength=2).astype(np.uint64))
    assert ran(k_enc, "fused_enc_kernel") and ran(k_dec, "fused_dec_kernel")
    nm, worst, err, rate8 = 0, 0.0, 0.0, 0.0
    for i in range(B):
        patches = crops(imgs[i:i + 1], P)
        ref = oracle_encoder(patches, "model_0", enc)
        n_i, w_i = check_symbols(sym_h[i], ref, patches, "model_0", enc)
        nm, worst = nm + n_i, max(worst, w_i)
        want = oracle_images(sym_h[i:i + 1], H, W, P, "model_0", dec)[0]
        e, r = check_recon(rec_f[i].cpu().numpy(), rec_u8[i].cpu().numpy(), want)
        err, rate8 = max(err, e), max(rate8, r)
    assert nm <= 1e-5 * sym_h.size
    # the streamed round trip from pinned host buffers is bit-identical to the device-resident calls
    h_imgs = torch.from_numpy(imgs).pin_memory()
    out = torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory()
    osym = torch.empty(tuple(sym.shape), dtype=torch.uint8).pin_memory()
    codec.roundtrip_images(h_imgs, P, out=out, out_symbols=osym)
    assert torch.equal(osym, sym.cpu()) and torch.equal(out, rec_u8.cpu())
    print(f"[A bench workload] {sym_h.shape[0] * sym_h.shape[1]} patches, {sym_h.size} symbols; mismatches {nm} "
          f"(max |fp64 logit| {worst:.2e}); recon max-abs {err:.2e}, u8 differing {rate8:.1e}; encode: {fmt(k_enc)}; "
          f"decode: {fmt(k_dec)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- B. wave and CTA-pair boundaries of the persistent kernels -------------------------------------------------------
# (variant, P, fused encoder pair, fused decoder pair)
@pytest.mark.parametrize("variant,P,enc_fused,dec_fused",
                         [("model_0", 128, True, True),                 # fused pairs around the u16 trunk
                          ("base_model/ch_128", 128, False, False),     # output-channel slices
                          ("model_1", 256, False, False),               # 3 -> 16 first layer, eight tile columns
                          ("base_model/input_256", 256, False, True),   # fused decoder at eight tile columns
                          ("model_3", 128, False, False),               # stride-2 80-channel quantiser, SIMT decode_4
                          ("model_2", 128, False, False)])              # stride-2 quantiser, decoder from symbols
def test_wave_and_pair_boundaries(variant, P, enc_fused, dec_fused):
    """A CTA pair takes patches pair0, pair0 + npairs, ... : patch counts of one patch, one pair, one wave of pairs minus /
    plus one patch, and two waves plus an odd tail, through encode_patches and decode_patches against the oracle.  Each
    count runs the prefix of one seeded batch, so one oracle pass covers them all.  On 8x8 maps two patches share a
    tile, so the largest counts also cross the first wave of the quantiser layer; the histogram the quantiser epilogue
    accumulates must equal np.bincount of the symbols it wrote at every count."""
    t0 = time.perf_counter()
    npairs = torch.cuda.get_device_properties(0).multi_processor_count // 2
    ns = [1, 2, 2 * npairs - 1, 2 * npairs, 2 * npairs + 1, 4 * npairs + 1, 4 * npairs + 3]
    codec, enc, dec = make_codec(variant, compute="tensor")
    patches = seeded_u8((max(ns), P, P, 3), 77)
    ref = oracle_encoder(patches, variant, enc)
    want = oracle_decoder(ref, variant, dec)
    nm, worst, err = 0, 0.0, 0.0
    for n in ns:
        codec.hist_reset()
        got = codec.encode_patches(patches[:n])
        assert np.array_equal(codec.hist_read(), np.bincount(got.reshape(-1), minlength=2).astype(np.uint64)), n
        n_i, w_i = check_symbols(got, ref[:n], patches[:n], variant, enc)
        nm, worst = nm + n_i, max(worst, w_i)
        e = float(np.abs(codec.decode_patches(ref[:n]) - want[:n]).max())
        assert e <= 1e-3, (n, e)
        err = max(err, e)
    k_enc = kernels_of(codec, lambda: codec.encode_patches(patches))
    k_dec = kernels_of(codec, lambda: codec.decode_patches(ref))
    assert ran(k_enc, "fused_enc_kernel") == enc_fused and ran(k_dec, "fused_dec_kernel") == dec_fused, (k_enc, k_dec)
    print(f"[B {variant}@{P}] n = {ns}: {sum(ns)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); recon max-abs "
          f"{err:.2e}; encode: {fmt(k_enc)}; decode: {fmt(k_dec)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


def test_float32_patches_past_one_wave():
    """float32 patches take the TMA-fed first layer with f32 windows (f16_first_s2_tma_kernel<true>) instead of the fused
    encoder: one wave of CTA pairs plus one patch, against the oracle."""
    t0 = time.perf_counter()
    n = torch.cuda.get_device_properties(0).multi_processor_count + 1
    codec, enc, dec = make_codec("model_0", compute="tensor")
    patches = seeded_u8((n, 128, 128, 3), 78)
    ref = oracle_encoder(patches, "model_0", enc)
    f32 = patches.astype(np.float32)
    sym = codec.encode_patches(f32)
    k = kernels_of(codec, lambda: codec.encode_patches(f32))
    assert ran(k, "f16_first_s2_tma_kernel<true>") and not ran(k, "fused_enc_kernel"), k
    nm, worst = check_symbols(sym, ref, patches, "model_0", enc)
    print(f"[B float32 patches] {n} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); encode: {fmt(k)}; "
          f"{time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- C. dispatch paths ------------------------------------------------------------------------------------------------
# (id, images H x W x count, byte offset of the device input, kernels the encoder must run, kernels it must not run,
#  kernels the decoder must run)
DISPATCH_CASES = [
    ("aligned", (512, 768, 4), 0, {"fused_enc_kernel"}, set(), {"fused_dec_kernel"}),
    ("offset1", (512, 768, 4), 1, {"f16_first_s2_kernel"}, {"fused_enc_kernel", "f16_first_s2_tma_kernel"}, {"fused_dec_kernel"}),
    ("offset4", (512, 768, 4), 4, {"f16_first_s2_kernel"}, {"fused_enc_kernel", "f16_first_s2_tma_kernel"}, {"fused_dec_kernel"}),
    ("offset8", (512, 768, 4), 8, {"f16_first_s2_kernel"}, {"fused_enc_kernel", "f16_first_s2_tma_kernel"}, {"fused_dec_kernel"}),
    # reflect-padded images; the 2- and 3-pixel sides reflect over many periods
    ("ragged2x130", (2, 130, 3), 0, {"f16_first_s2_kernel"}, {"fused_enc_kernel"}, {"fused_dec_kernel"}),
    ("ragged3x3", (3, 3, 3), 0, {"f16_first_s2_kernel"}, {"fused_enc_kernel"}, {"fused_dec_kernel"}),
    ("ragged64x300", (64, 300, 2), 0, {"f16_first_s2_kernel"}, {"fused_enc_kernel"}, {"fused_dec_kernel"}),
    ("ragged129x385", (129, 385, 2), 0, {"f16_first_s2_kernel"}, {"fused_enc_kernel"}, {"fused_dec_kernel"}),
    ("ragged1356x2040", (1356, 2040, 1), 0, {"f16_first_s2_kernel"}, {"fused_enc_kernel"}, {"fused_dec_kernel"}),
]


@pytest.mark.parametrize("case", DISPATCH_CASES, ids=[c[0] for c in DISPATCH_CASES])
def test_dispatch_paths_against_oracle(case):
    """model_0 @128 in tensor mode on u8 images on the device: the kernels each input selects, by name, and its symbols and
    reconstruction against the oracle (crop with np.pad 'reflect', decode, stitch, crop).  A misaligned input cannot be
    read by TMA and takes the windowed first layer; it must agree with the aligned call, and so must a decode into a
    misaligned output."""
    t0 = time.perf_counter()
    name, (H, W, B), off, enc_want, enc_forbid, dec_want = case
    P = 128
    codec, enc, dec = make_codec("model_0", compute="tensor")
    imgs = seeded_u8((B, H, W, 3), 100 + H + W)
    d_imgs = device_view(imgs, off)
    sym = codec.encode_images(d_imgs, P)
    k_enc = kernels_of(codec, lambda: codec.encode_images(d_imgs, P))
    assert all(ran(k_enc, k) for k in enc_want) and not any(ran(k_enc, k) for k in enc_forbid), fmt(k_enc)
    sym_h = sym.cpu().numpy()
    patches = crops(imgs, P)
    nm, worst = check_symbols(sym_h, oracle_encoder(patches, "model_0", enc), patches, "model_0", enc)
    rec_f = codec.decode_images(sym, H, W, P, out_dtype=np.float32)
    k_dec = kernels_of(codec, lambda: codec.decode_images(sym, H, W, P, out_dtype=np.float32))
    assert all(ran(k_dec, k) for k in dec_want), fmt(k_dec)
    rec_u8 = codec.decode_images(sym, H, W, P)
    want = oracle_images(sym_h, H, W, P, "model_0", dec)
    err, rate8 = check_recon(rec_f.cpu().numpy(), rec_u8.cpu().numpy(), want)
    if off:
        # the aligned call: the same symbols but where both paths sit in the dead zone, and the same reconstruction
        aligned = codec.encode_images(device_view(imgs, 0), P).cpu().numpy()
        check_symbols(sym_h, aligned.reshape(-1, 8, 8, 64), patches, "model_0", enc)
        out8 = device_view(np.zeros((B, H, W, 3), np.uint8), off)
        codec.decode_images(sym, H, W, P, out=out8)
        assert torch.equal(out8, rec_u8)
        if off % 4 == 0:
            outf = device_view(np.zeros((B, H, W, 3), np.float32), off, torch.float32)
            codec.decode_images(sym, H, W, P, out=outf)
            assert torch.equal(outf, rec_f)
    print(f"[C {name}] {B} x {H}x{W}, {len(patches)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); recon max-abs "
          f"{err:.2e}, u8 differing {rate8:.1e}; encode: {fmt(k_enc)}; decode: {fmt(k_dec)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


@pytest.mark.parametrize("P", [32, 64, 96, 128, 160, 192, 256, 320, 512])
def test_patch_size_sweep(P):
    """model_0 on exact-grid u8 images (2 x 2P x 3P): a patch size the fp32 path accepts must run in tensor mode too,
    whichever kernels that selects, and match the oracle.  An error from a tensor kernel that was selected is a failure."""
    t0 = time.perf_counter()
    codec, enc, dec = make_codec("model_0", compute="fp32")
    H, W = 2 * P, 3 * P
    imgs = seeded_u8((2, H, W, 3), 200 + P)
    try:
        codec.encode_images(imgs, P)
    except (ValueError, T.TicError) as e:
        codec.close()
        pytest.skip(f"P = {P} is not supported by the fp32 path either: {e}")
    codec.set_compute("tensor")
    d_imgs = torch.from_numpy(imgs).cuda()
    sym = codec.encode_images(d_imgs, P)
    k_enc = kernels_of(codec, lambda: codec.encode_images(d_imgs, P))
    sym_h = sym.cpu().numpy()
    patches = crops(imgs, P)
    nm, worst = check_symbols(sym_h, oracle_encoder(patches, "model_0", enc), patches, "model_0", enc)
    rec_f = codec.decode_images(sym, H, W, P, out_dtype=np.float32)
    k_dec = kernels_of(codec, lambda: codec.decode_images(sym, H, W, P, out_dtype=np.float32))
    rec_u8 = codec.decode_images(sym, H, W, P)
    err, rate8 = check_recon(rec_f.cpu().numpy(), rec_u8.cpu().numpy(), oracle_images(sym_h, H, W, P, "model_0", dec))
    # the fused pairs take exactly the patch sizes their tiling covers
    assert ran(k_enc, "fused_enc_kernel") == (P % 64 == 0 and P // 32 <= 8), fmt(k_enc)
    print(f"[C P={P}] {len(patches)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); recon max-abs {err:.2e}, "
          f"u8 differing {rate8:.1e}; encode: {fmt(k_enc)}; decode: {fmt(k_dec)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


@pytest.mark.parametrize("mean,fused", [(-768.0, True), (1023.0, True), (-769.0, False), (1024.0, False),
                                        (-1000.0, False), (1500.0, False)])
def test_channel_means_around_the_fused_range(mean, fused):
    """The fused encoder works on the exact integers x - round(mean), which must stay in its fp16 range: means that round
    into [-768, 1023] run fused_enc_kernel, others the first-layer + u16 kernels.  Either way tensor-mode encoding of
    exact-grid u8 images must succeed and match the oracle."""
    t0 = time.perf_counter()
    means = np.full(3, mean, np.float32)
    enc, dec = params_for("model_0", "fanin")
    codec = T.Codec("model_0", quan_scale=2, mean=means, std=STD, enc_params=enc, dec_params=dec, compute="tensor")
    imgs = seeded_u8((4, 512, 768, 3), 300)
    d_imgs = torch.from_numpy(imgs).cuda()
    sym = codec.encode_images(d_imgs, 128)
    codec.check_status()
    k = kernels_of(codec, lambda: codec.encode_images(d_imgs, 128))
    assert ran(k, "fused_enc_kernel") == fused and (fused or ran(k, "f16_first_s2_tma_kernel<false>")), fmt(k)
    patches = crops(imgs, 128)
    nm, worst = check_symbols(sym.cpu().numpy(), oracle_encoder(patches, "model_0", enc, means), patches, "model_0", enc,
                              means)
    print(f"[C mean {mean}] {len(patches)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); encode: {fmt(k)}; "
          f"{time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- D. chunk boundaries ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [1, 7, 23, 25, 47, 4096])
def test_chunk_boundaries(chunk):
    """set_chunk_patches(c) with host and device buffers: image calls run whole images per chunk (at least one), patch
    calls cut the 24-patch images anywhere.  encode / decode / round trip results are bit-identical to the one-chunk
    call, whose symbols and reconstruction match the oracle."""
    t0 = time.perf_counter()
    B, H, W, P = 5, 512, 768, 128
    codec, enc, dec = make_codec("model_0", compute="tensor")
    imgs = seeded_u8((B, H, W, 3), 400)
    patches = crops(imgs, P)
    sym = codec.encode_images(imgs, P)
    rec_u8 = codec.decode_images(sym, H, W, P)
    rec_f = codec.decode_images(sym, H, W, P, out_dtype=np.float32)
    nm, worst = check_symbols(sym, oracle_encoder(patches, "model_0", enc), patches, "model_0", enc)
    err, rate8 = check_recon(rec_f, rec_u8, oracle_images(sym, H, W, P, "model_0", dec))
    psym = sym.reshape(-1, 8, 8, 64)
    prec = codec.decode_patches(psym)
    codec.set_chunk_patches(chunk)
    for dev in (False, True):
        put = (lambda a: torch.from_numpy(a).cuda()) if dev else (lambda a: a)
        get = (lambda t: t.cpu().numpy()) if dev else (lambda a: a)
        assert np.array_equal(get(codec.encode_images(put(imgs), P)), sym)
        assert np.array_equal(get(codec.decode_images(put(sym), H, W, P)), rec_u8)
        assert np.array_equal(get(codec.decode_images(put(sym), H, W, P, out_dtype=np.float32)), rec_f)
        r, s = codec.roundtrip_images(put(imgs), P)
        assert np.array_equal(get(s), sym) and np.array_equal(get(r), rec_u8)
        assert np.array_equal(get(codec.encode_patches(put(patches))), psym)
        assert np.array_equal(get(codec.decode_patches(put(psym))), prec)
    print(f"[D chunk {chunk}] {len(patches)} patches; mismatches {nm} (max |fp64 logit| {worst:.2e}); recon max-abs "
          f"{err:.2e}, u8 differing {rate8:.1e}; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- E. quan_scale > 2 in tensor mode ---------------------------------------------------------------------------------
@pytest.mark.parametrize("variant,q", [pytest.param("model_0", q, id=str(q)) for q in (3, 4, 16, 255, 256)] +
                         [pytest.param("model_3", q, id=f"model_3-{q}") for q in (3, 16)])
def test_quan_scale_in_tensor_mode(variant, q):
    """The quantiser epilogue, the general (q != 2) histogram and the q-entry inverse-sigmoid table of the tensor path:
    model_0's stride-1 64-channel quantiser, and model_3's stride-2 80-channel one (8 epilogue warps), whose decoder
    reads the table on the CUDA cores.
    A symbol may differ from the oracle's by one where the fp64 value sigmoid(logit) * (q - 1) is within fp32 noise of a
    half-integer: the logit's accumulation error (4e-6 of the largest logit, as for q = 2) times the sigmoid's slope
    (at most (q - 1) / 4), plus a few fp32 ulps of sigmoid * (q - 1)."""
    t0 = time.perf_counter()
    codec, enc, dec = make_codec(variant, q=q, compute="tensor")
    patches = seeded_u8((48, 128, 128, 3), 500 + q)
    codec.hist_reset()
    sym = codec.encode_patches(patches)
    assert np.array_equal(codec.hist_read(), np.bincount(sym.reshape(-1), minlength=q).astype(np.uint64))
    ref = oracle_encoder(patches, variant, enc, q=q)
    d = np.abs(sym.astype(np.int32) - ref.astype(np.int32))
    assert d.max() <= 1
    nm, dist, bound = int((d != 0).sum()), 0.0, 0.0
    if nm:
        l64 = logits64(patches, variant, enc, MEAN, STD)
        o = (q - 1) / (1 + np.exp(-l64[d != 0]))
        dist = float(np.abs(o - np.floor(o) - 0.5).max())
        bound = (q - 1) * 1e-6 * float(np.abs(l64).max()) + 4 * np.spacing(np.float32(q - 1)).item()
        assert dist <= bound, f"a mismatch {dist:.3e} from a half-integer, bound {bound:.3e}"
    rec = codec.decode_patches(ref)
    err = float(np.abs(rec - oracle_decoder(ref, variant, dec, q=q)).max())
    assert err <= 1e-3
    print(f"[E {variant} q={q}] {len(patches)} patches, {ref.size} symbols; mismatches {nm} (|d| <= 1, max distance from a "
          f"half-integer {dist:.2e}, bound {bound:.2e}); recon max-abs {err:.2e}; {time.perf_counter() - t0:.1f} s")
    codec.close()
