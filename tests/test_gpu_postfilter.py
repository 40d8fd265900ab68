"""-m gpu parity of the rmbe de-blocking post-filter on whole images (Codec.postfilter_images, rmbe.rmbe) against the CPU
oracle O.rmbe, on every tile geometry and first-layer dispatch path, across chunk splits, host and device buffers, and
BASELINE config 5 at the benchmark's 2048x1536.

Bars (every case prints the three errors):
- float: max |gpu - oracle32| <= 2e-3 after both passes (3e-3 where the decoder runs first);
- fp64: max |gpu - f64| <= 4 max |oracle32 - f64| + 4e-4, with f64 the same two passes evaluated in float64 (arbiter64);
- pixels outside every tile of both passes are bit-identical to the input (the tile grids of submit/2/rmbe/rmbe.py:70-111).
Tensor-mode cases name the first-layer kernel the input selects: the TMA-fed f16_first_s2_tma_kernel<true> when the
row pitch (W * 12 bytes) and the base address are multiples of 16 bytes, else the gather kernel f16_first_s2_kernel."""
import time

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
import tf_image_compression_b200 as T
from gpu_common import MEAN, PM, PS, STD, device_view, fmt, in_tiles, kernels_of, make_codec, oracle32, post_params, ran

pytestmark = pytest.mark.gpu

MODES = ["fp32", "tensor"]
P, OFF = 128, 64  # rmbe tile edge and grid offset (submit/2/rmbe/rmbe.py:12,16)

_cache = {}


def cached(key, fn):
    """The oracle results of one input are shared by the compute modes that check against them."""
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def pf_codec(mode, name="rmbe", pp=None):
    codec, _, _ = make_codec("model_1", compute=mode)
    codec.set_postfilter(post_params(name) if pp is None else pp, PM, PS, name=name)
    return codec


def images(B, H, W, seed):
    """[B,H,W,3] float32: a natural image (O.synthetic_image), continuous uniform noise, and a contrast-stretched natural
    image with large areas of exact 0 and 255, in turn."""
    rs = np.random.RandomState(seed)
    out = []
    for i in range(B):
        nat = O.synthetic_image(H, W, seed + i).astype(np.float32)
        kind = i % 3 if B > 1 else 0
        if kind == 1:
            out.append(rs.uniform(0.0, 255.0, size=(H, W, 3)).astype(np.float32))
        elif kind == 2:
            out.append(np.clip((nat - 128.0) * 4.0 + 128.0, 0.0, 255.0).astype(np.float32))
        else:
            out.append(nat)
    return np.stack(out)


def tile_grids(H, W):
    """(oy, ox, rows, cols) of pass 1 (rmbe_height) and pass 2 (rmbe_width), submit/2/rmbe/rmbe.py:70-111."""
    return ((0, OFF, H // P, max(0, (W - OFF) // P)), (OFF, 0, max(0, (H - OFF) // P), W // P))


def untouched(H, W):
    """[H,W] mask of the pixels outside every tile of both passes."""
    m = np.ones((H, W), bool)
    for oy, ox, hn, wn in tile_grids(H, W):
        m[oy:oy + hn * P, ox:ox + wn * P] = False
    return m


def arbiter64(img, name, pp, mean=PM, std=PS):
    """O.rmbe's two passes in float64: normalisation, the layers and the denormalisation + clip in float64, and the image
    kept in float64 between the passes.  The weights, means and stds are the float32 values the codec holds."""
    m64, s64 = np.asarray(mean, np.float32).astype(np.float64), np.asarray(std, np.float32).astype(np.float64)

    def run(t):
        y = O.run_layers((t - m64) / s64, O.POSTFILTERS[name], 3, pp, dtype=torch.float64)
        return np.clip(y * s64 + m64, 0.0, 255.0)

    image = np.array(img, dtype=np.float64, copy=True)
    H, W, _ = image.shape
    for oy, ox, hn, wn in tile_grids(H, W):
        if hn * wn == 0:
            continue
        tiles = np.stack([image[oy + i * P:oy + (i + 1) * P, ox + j * P:ox + (j + 1) * P] for i in range(hn) for j in range(wn)])
        new = in_tiles(run, tiles)
        for i in range(hn):
            for j in range(wn):
                image[oy + i * P:oy + (i + 1) * P, ox + j * P:ox + (j + 1) * P] = new[i * wn + j]
    return image


def check_filtered(tag, got, inp, want32, want64=None, bar=2e-3):
    """The float bar against the oracle, the fp64 rule where an fp64 result is given, and bit-identical pixels outside
    the tiles.  Returns (|gpu - oracle32|, |gpu - f64|, |oracle32 - f64|) as max-abs over the batch."""
    got, inp = np.asarray(got), np.asarray(inp)
    e32 = float(np.abs(got - want32).max())
    e64 = r64 = float("nan")
    if want64 is not None:
        e64, r64 = float(np.abs(got - want64).max()), float(np.abs(want32 - want64).max())
    print(f"  [{tag}] |gpu-oracle32| {e32:.3e}  |gpu-f64| {e64:.3e}  |oracle32-f64| {r64:.3e}")
    mask = untouched(got.shape[1], got.shape[2])
    assert np.array_equal(got[:, mask].view(np.uint32), inp[:, mask].view(np.uint32)), f"{tag}: a pixel outside the tiles changed"
    assert e32 <= bar, f"{tag}: |gpu - oracle32| {e32:.3e} > {bar}"
    if want64 is not None:
        assert e64 <= 4.0 * r64 + 4e-4, f"{tag}: |gpu - f64| {e64:.3e} > 4 x {r64:.3e} + 4e-4"
    return e32, e64, r64


def first_layer_check(mode, names, want):
    """The first-layer kernel by name: want = 'tma' | 'gather' (tensor mode), CUDA-core kernels only in fp32 mode."""
    if mode == "fp32":
        assert ran(names, "conv3x3_simt_kernel"), fmt(names)
        assert not any(n.startswith(("f16_", "u16", "umma", "fused")) for n in names), fmt(names)
    elif mode == "tensor":
        tma, gather = ran(names, "f16_first_s2_tma_kernel<true>"), ran(names, "f16_first_s2_kernel")
        assert (tma, gather) == ((True, False) if want == "tma" else (False, True)), fmt(names)
    else:  # 3xtf32: the f32 image is read by the CUDA-core first layer, the 32/64-channel layers run on umma_conv_kernel
        assert ran(names, "conv3x3_simt_kernel") and ran(names, "umma_conv_kernel"), fmt(names)
        assert not any(n.startswith(("f16_", "u16")) for n in names), fmt(names)


# ---- A. tile geometries and first-layer dispatch paths ---------------------------------------------------------------
# (id, B, H, W, byte offset of a device input (None: host array), tensor-mode first layer, fp64 arbiter)
GEOMETRY_CASES = [
    ("tma", 2, 384, 448, None, "tma", True),            # 9 + 6 tiles per image
    ("ragged", 3, 200, 300, None, "tma", True),         # H, W not multiples of 128; W % 4 == 0
    ("gather_w", 2, 257, 450, None, "gather", True),    # W * 12 % 16 == 8: no tensor map for this row pitch
    ("gather_off", 4, 512, 768, 4, "gather", True),     # device input 4 bytes past a 16-byte boundary
    ("pass1_only", 1, 128, 192, None, "tma", True),     # pass 2 has no tiles
    ("pass2_only", 1, 192, 128, None, "tma", True),     # pass 1 has no tiles
    ("none_100", 1, 100, 100, None, None, False),       # no tiles at all
    ("none_63x4000", 1, 63, 4000, None, None, False),
    ("big_odd", 1, 1356, 2041, None, "gather", True),   # 150 + 150 tiles on the gather path
]
GEOMETRY_PARAMS = [pytest.param(c, m, id=f"{c[0]}-{m}") for c in GEOMETRY_CASES for m in MODES] + \
                  [pytest.param(GEOMETRY_CASES[0], "3xtf32", id="tma-3xtf32")]


@pytest.mark.parametrize("case,mode", GEOMETRY_PARAMS)
def test_geometry_against_oracle(case, mode):
    """postfilter_images on one batch per geometry: the float bar, the fp64 rule and untouched pixels outside the tiles.
    gather_off: the input is a device tensor 4 bytes past an aligned address, which the tensor map cannot take, so the
    gather kernel runs.  Its result must be BITWISE equal to the aligned call's (TMA) result: both builders produce the
    same fp16 pair per pixel — the gather builder divides (x - mean) / std, the TMA builder forms the quotient from the
    correctly rounded reciprocal with one FMA residual correction, and the two agree on every float in [0, 255] for these
    means and stds — and the MMAs and epilogues that follow are the same instructions.  Geometries without tiles must
    launch nothing and leave the image bit-identical."""
    t0 = time.perf_counter()
    name_id, B, H, W, off, path, use64 = case
    pp = post_params()
    codec = pf_codec(mode)
    inp = images(B, H, W, 1000 + H + W)
    want32 = cached(("rmbe", name_id, "32"), lambda: np.stack([oracle32(im, "rmbe", pp) for im in inp]))
    want64 = cached(("rmbe", name_id, "64"), lambda: np.stack([arbiter64(im, "rmbe", pp) for im in inp])) if use64 else None
    if off is None:
        got = inp.copy()
        codec.postfilter_images(got)
        scratch = inp.copy()
    else:
        d = device_view(inp, off, torch.float32)
        codec.postfilter_images(d)
        got = d.cpu().numpy()
        scratch = device_view(inp, off, torch.float32)
    codec.check_status()
    names = kernels_of(codec, lambda: codec.postfilter_images(scratch))
    tiles = sum(hn * wn for _, _, hn, wn in tile_grids(H, W))
    if tiles == 0:
        assert names == set() and np.array_equal(got.view(np.uint32), inp.view(np.uint32))
        print(f"[A {name_id} {mode}] {B} x {H}x{W}: no tiles, no launches, image unchanged; {time.perf_counter() - t0:.1f} s")
        codec.close()
        return
    first_layer_check(mode, names, path)
    e32, e64, r64 = check_filtered(f"{name_id} {mode}", got, inp, want32, want64)
    if off is not None:
        aligned = torch.from_numpy(inp).cuda()
        codec.postfilter_images(aligned)
        k_al = kernels_of(codec, lambda: codec.postfilter_images(torch.from_numpy(inp).cuda()))
        if mode == "tensor":
            assert ran(k_al, "f16_first_s2_tma_kernel<true>"), fmt(k_al)
        assert np.array_equal(aligned.cpu().numpy().view(np.uint32), got.view(np.uint32)), \
            f"misaligned != aligned, max-abs {float(np.abs(aligned.cpu().numpy() - got).max()):.3e}"
    print(f"[A {name_id} {mode}] {B} x {H}x{W}, {tiles} tiles per image; |gpu-oracle32| {e32:.2e}, |gpu-f64| {e64:.2e}, "
          f"|oracle32-f64| {r64:.2e}; kernels: {fmt(names)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- B. chunk splits, host vs device, batch vs single image, repetition -----------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_chunk_splits_and_buffers_are_bit_identical(mode):
    """5 x 384x448 images, 9 pass-1 and 6 pass-2 tiles each.  set_chunk_patches(c) for c = 1, 9, 18, 27, 4096 (images per
    chunk 1, 1, 2, 3, all; c = 1 gives one image of more tiles than the chunk) on host arrays (staged chunk by chunk) and
    on device tensors (chunks after the first address their images through the patch offset n0 = u0 * tiles and, in
    tensor mode, the image dimension of the tensor map) gives the bytes of the one-chunk call.  So do each image alone
    ([H,W,3]) and a repeated call; the fp16 range guard stays clean; the one-chunk call meets the float bar."""
    t0 = time.perf_counter()
    B, H, W = 5, 384, 448
    pp = post_params()
    codec = pf_codec(mode)
    inp = images(B, H, W, 2000)
    ref = inp.copy()
    codec.postfilter_images(ref)
    e32, _, _ = check_filtered(f"chunks {mode}", ref, inp, np.stack([oracle32(im, "rmbe", pp) for im in inp]))
    again = inp.copy()
    codec.postfilter_images(again)
    assert np.array_equal(again.view(np.uint32), ref.view(np.uint32)), "repeated call differs"
    for i in range(B):
        one = inp[i].copy()
        assert codec.postfilter_images(one) is one
        assert np.array_equal(one.view(np.uint32), ref[i].view(np.uint32)), f"image {i} alone differs from the batch"
    for c in (1, 9, 18, 27, 4096):
        codec.set_chunk_patches(c)
        h = inp.copy()
        codec.postfilter_images(h)
        assert np.array_equal(h.view(np.uint32), ref.view(np.uint32)), f"host buffers, chunk {c}"
        d = torch.from_numpy(inp).cuda()
        codec.postfilter_images(d)
        assert np.array_equal(d.cpu().numpy().view(np.uint32), ref.view(np.uint32)), f"device buffers, chunk {c}"
    codec.check_status()
    print(f"[B chunks {mode}] {B} x {H}x{W}; |gpu-oracle32| {e32:.2e}; host, device, per image, repeated and chunks "
          f"1/9/18/27/4096 bit-identical; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- C. the stride-1 post-filter rmbe_model_1 on images ---------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B,H,W", [(2, 384, 448), (1, 257, 450)])
def test_rmbe_model_1_images(B, H, W, mode):
    """rm_block_effect/model_1 (four stride-1 convs) through postfilter_images.  In tensor mode its first layer is the
    im2col kernel f16_first_kernel<1> reading f32 pixels through the shifted tile grid, and its 32 -> 3 last layer into
    the image runs on the CUDA cores (conv3x3_simt_kernel): the pair-plane kernels write an image only from a transposed
    3-channel layer.  Both read and write through the tile grid."""
    t0 = time.perf_counter()
    pp = post_params("rmbe_model_1")
    codec = pf_codec(mode, "rmbe_model_1", pp)
    inp = images(B, H, W, 3000 + W)
    want32 = cached(("m1", H, W, "32"), lambda: np.stack([oracle32(im, "rmbe_model_1", pp) for im in inp]))
    want64 = cached(("m1", H, W, "64"), lambda: np.stack([arbiter64(im, "rmbe_model_1", pp) for im in inp]))
    got = inp.copy()
    codec.postfilter_images(got)
    codec.check_status()
    scratch = inp.copy()
    names = kernels_of(codec, lambda: codec.postfilter_images(scratch))
    if mode == "tensor":
        assert ran(names, "f16_first_kernel<1>") and ran(names, "conv3x3_simt_kernel"), fmt(names)
    else:
        assert not any(n.startswith(("f16_", "u16", "umma", "fused")) for n in names), fmt(names)
    e32, e64, r64 = check_filtered(f"model_1 {B}x{H}x{W} {mode}", got, inp, want32, want64)
    print(f"[C rmbe_model_1 {mode}] {B} x {H}x{W}; |gpu-oracle32| {e32:.2e}, |gpu-f64| {e64:.2e}, |oracle32-f64| {r64:.2e}; "
          f"kernels: {fmt(names)}; {time.perf_counter() - t0:.1f} s")
    codec.close()


# ---- D. the Python surface ----------------------------------------------------------------------------------------------
def test_rmbe_surface_and_shape_validation():
    """rmbe.rmbe keeps the reference's contract (submit/2/rmbe/rmbe.py:15-25): a float32 C-contiguous array is filtered in
    place and returned; u8 or float64 input gives a new float32 array and is left alone; device tensors are filtered in
    place.  Anything but [B,H,W,3] / [H,W,3] is a ValueError before the library is called, for host arrays and device
    tensors alike (the library reads and writes H*W*3 floats per image)."""
    codec = pf_codec("fp32")
    T.rmbe.bind(codec)
    try:
        base = images(1, 192, 320, 4000)[0]
        want = base.copy()
        codec.postfilter_images(want)
        assert not np.array_equal(want, base)
        f = base.copy()
        assert T.rmbe.rmbe(f) is f and np.array_equal(f, want)
        for src in (np.round(base).astype(np.uint8), base.astype(np.float64)):
            keep = src.copy()
            out = T.rmbe.rmbe(src)
            assert out is not src and out.dtype == np.float32 and np.array_equal(src, keep)
            w = src.astype(np.float32)
            codec.postfilter_images(w)
            assert np.array_equal(out, w)
        d = torch.from_numpy(base).cuda()
        assert T.rmbe.rmbe(d) is d and np.array_equal(d.cpu().numpy(), want)
        for shape in [(192, 320), (2, 192, 320, 4), (2, 192, 320, 1), (192, 320, 4), (1, 2, 192, 320, 3)]:
            for x in (np.zeros(shape, np.float32), torch.zeros(shape, dtype=torch.float32, device="cuda")):
                with pytest.raises(ValueError):
                    codec.postfilter_images(x)
                with pytest.raises(ValueError):
                    T.rmbe.rmbe(x)
        codec.check_status()
    finally:
        T.rmbe.bind(None)
        codec.close()


# ---- E. BASELINE config 5 at the benchmark's size -------------------------------------------------------------------------
def oracle_decode(sym, H, W, dec, mean, std):
    """model_1 decoder (P = 256) of one image's [48, 16, 16, 64] symbols, stitched: [H,W,3] float32."""
    rec = np.concatenate([O.decoder(sym[i:i + 8], "model_1", dec, mean, std, 2) for i in range(0, len(sym), 8)])
    return O.concat_patches(list(rec), H, W, 256)


def check_cfg5(tag, codec, sym, dec, pp, post_mean, post_std, key):
    """decode_images -> postfilter_images -> round_u8 on device tensors of 2 x 2048x1536 images, per image against the
    oracle's decode -> O.rmbe -> np.around: the decode within 1e-3, the filtered image within 3e-3, and the u8 image at
    most one grey level off, only where the oracle's float value is within (the measured float error + 1e-4) of a .5
    boundary.  Returns (decode error, filtered error, u8 values that differ)."""
    H, W = 1536, 2048
    d_sym = torch.from_numpy(sym).cuda()
    img = codec.decode_images(d_sym, H, W, 256, out_dtype=np.float32)
    dec_gpu = img.cpu().numpy()
    codec.postfilter_images(img)
    out8 = codec.round_u8(img).cpu().numpy()
    codec.check_status()
    got = img.cpu().numpy()
    scratch = torch.from_numpy(dec_gpu).cuda()
    names = kernels_of(codec, lambda: codec.postfilter_images(scratch))
    first_layer_check(codec.compute, names, "tma")
    e_dec = e_f = 0.0
    n8 = 0
    for i in range(len(sym)):
        want_dec = cached((key, i, "dec"), lambda: oracle_decode(sym[i], H, W, dec, MEAN, STD))
        want = cached((key, i, "rmbe"), lambda: oracle32(want_dec, "rmbe", pp, post_mean, post_std))
        e_dec = max(e_dec, float(np.abs(dec_gpu[i] - want_dec).max()))
        ei = float(np.abs(got[i] - want).max())
        assert np.array_equal(got[i][untouched(H, W)], dec_gpu[i][untouched(H, W)])
        d = np.abs(out8[i].astype(np.int32) - O.around_u8(want).astype(np.int32))
        near = np.abs(want - np.floor(want) - 0.5) <= ei + 1e-4
        assert d.max() <= 1 and not (d[~near] != 0).any(), f"{tag} image {i}: u8 differs away from a .5 boundary"
        e_f, n8 = max(e_f, ei), n8 + int((d != 0).sum())
    print(f"  [{tag}] decode |gpu-oracle32| {e_dec:.3e}; decode + rmbe |gpu-oracle32| {e_f:.3e}; u8 differing {n8}; "
          f"kernels: {fmt(names)}")
    assert e_dec <= 1e-3 and e_f <= 3e-3, (e_dec, e_f)
    return e_dec, e_f, n8


@pytest.mark.parametrize("mode", MODES)
def test_cfg5_benchmark_scale(mode):
    """Config 5 as bench.py times it (model_1 decode at P = 256 -> stitch -> rmbe -> np.around, 356 filter tiles per
    image) on 2 x 2048x1536 images: once with the fan-in weights of the tests above, and once with the weights bench.py
    itself runs (Codec(..., seed=1234) and set_postfilter() defaults), the oracle given the same reference_init arrays."""
    t0 = time.perf_counter()
    sym = np.random.RandomState(8).randint(0, 2, size=(2, 48, 16, 16, 64)).astype(np.uint8)
    codec, _, dec = make_codec("model_1", compute=mode)
    pp = post_params()
    codec.set_postfilter(pp, PM, PS)
    check_cfg5(f"cfg5 fan-in {mode}", codec, sym, dec, pp, PM, PS, "cfg5_fanin")
    codec.close()
    codec = T.Codec("model_1", quan_scale=2, mean=MEAN, std=STD, compute=mode, seed=1234)
    codec.set_postfilter()
    dec = T.reference_init(codec.dec_layers, 1234 + 1)
    pp = T.reference_init(codec.post_layers, 4321)
    check_cfg5(f"cfg5 bench weights {mode}", codec, sym, dec, pp, MEAN, STD, "cfg5_bench")
    codec.close()
    print(f"[E cfg5 {mode}] 2 x 2048x1536; {time.perf_counter() - t0:.1f} s")
