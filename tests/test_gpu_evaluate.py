"""-m gpu: rate-distortion evaluation on the device (Codec.evaluate_images / entry.evaluate) against the file flow it
replaces (entry.compress -> entry.uncompress -> evaluate.py's formulas), the entropy stage and the decoder.  Every
comparison is exact."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
import tf_image_compression_b200 as T
from tf_image_compression_b200 import _lib as L
from tf_image_compression_b200 import entry
from gpu_common import MEAN, STD, make_codec, params_for

pytestmark = pytest.mark.gpu


def _sse(a, b):
    d = a.astype(np.int64) - b.astype(np.int64)
    return int((d * d).sum())


def _prob(codec, images, P):
    codec.hist_reset()
    for im in images:
        codec.encode_images(im[None], P)
    counts = codec.hist_read().astype(np.float64)
    return counts / counts.sum()


@pytest.mark.parametrize("mode", ["fp32", "tensor"])
def test_against_the_file_flow(mode, tmp_path):
    """model_0@128: 2048x1536 (fused TMA encoder in tensor mode), 768x512, 300x200 (reflect padding) and 128x128 (one
    patch: a plain stream, not the segmented container)."""
    codec, _, _ = make_codec("model_0", "fanin", compute=mode)
    shapes = [(1536, 2048), (512, 768), (200, 300), (512, 768), (128, 128)]
    images = [O.synthetic_image(h, w, 40 + i) for i, (h, w) in enumerate(shapes)]
    names = [f"img_{i}" for i in range(len(images))]
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=128)
    prob = _prob(codec, images, 128)
    files = entry.compress(codec, images, names, cfg, prob, str(tmp_path / "enc"), coder="host")
    recs = entry.uncompress(codec, str(tmp_path / "enc"), cfg, prob)
    sizes = [n for _, n in files]
    rec_list = [recs[n] for n in names]
    res = entry.evaluate(codec, images, cfg, prob)
    assert res["code_bytes"].tolist() == sizes
    assert res["sq_err"].tolist() == [_sse(a, b) for a, b in zip(images, rec_list)]
    assert res["bpp"] == entry.bpp(sizes, images)
    assert res["psnr"] == entry.psnr(images, rec_list)
    codec.close()


@pytest.mark.parametrize("variant,P", [("model_1", 256), ("base_model/reduced_btn_32", 128), ("model_3", 128),
                                       ("model_2", 128)])
def test_other_variants(variant, P):
    """model_1 at P = 256, a 32-channel bottleneck whose decoder tail is not the fused pair, and the submitted codecs
    model_3 (80-channel bottleneck, CUDA-core decode_4) and model_2 (stride-2 quantiser, decoder from symbols): lengths
    equal entropy_encode's, squared errors equal those of decode_images."""
    codec, _, _ = make_codec(variant, "fanin", compute="tensor")
    batch = np.stack([O.synthetic_image(512, 768, 60 + i) for i in range(3)])
    small = O.synthetic_image(200, 300, 70)[None]
    cum = entry.cum_freq_table(_prob(codec, list(batch), P), 4096)
    for imgs in (batch, small):
        sym = codec.encode_images(imgs, P)
        _, nbytes = codec.entropy_encode(sym, cum)
        rec = codec.decode_images(sym, imgs.shape[1], imgs.shape[2], P)
        cb, se, _ = codec.evaluate_images(imgs, P, cum)
        assert cb.tolist() == nbytes.tolist()
        assert se.tolist() == [_sse(a, b) for a, b in zip(imgs, rec)]
    codec.close()


def test_host_and_device_buffers_and_reconstruction():
    codec, _, _ = make_codec("model_0", "fanin", compute="tensor")
    imgs = np.stack([O.synthetic_image(512, 768, 80 + i) for i in range(3)])
    cum = entry.cum_freq_table(_prob(codec, list(imgs), 128), 4096)
    rec_rt, _ = codec.roundtrip_images(imgs, 128, want_symbols=False)
    out = np.zeros_like(imgs)
    cb_h, se_h, r = codec.evaluate_images(imgs, 128, cum, out=out)
    assert r is out and np.array_equal(out, rec_rt)
    assert cb_h.dtype == np.int64 and se_h.dtype == np.uint64
    assert se_h.tolist() == [_sse(a, b) for a, b in zip(imgs, rec_rt)]
    cb_n, se_n, r_n = codec.evaluate_images(imgs, 128, cum)
    assert r_n is None and np.array_equal(cb_n, cb_h) and np.array_equal(se_n, se_h)
    pinned = torch.from_numpy(imgs).pin_memory()
    cb_p, se_p, _ = codec.evaluate_images(pinned, 128, cum)
    assert np.array_equal(cb_p, cb_h) and np.array_equal(se_p, se_h)
    d_imgs = torch.from_numpy(imgs).cuda()
    d_out = torch.zeros_like(d_imgs)
    cb_d, se_d, _ = codec.evaluate_images(d_imgs, 128, cum, out=d_out)
    cb_d2, se_d2, _ = codec.evaluate_images(d_imgs, 128, cum)
    codec.check_status()
    assert cb_d.is_cuda and cb_d.dtype == torch.int64 and se_d.dtype == torch.int64
    for cb, se in ((cb_d, se_d), (cb_d2, se_d2)):
        assert cb.cpu().tolist() == cb_h.tolist() and se.cpu().tolist() == se_h.tolist()
    assert np.array_equal(d_out.cpu().numpy(), rec_rt)
    codec.close()


@pytest.mark.parametrize("chunk", [24, 48])
def test_chunk_splits_and_repeated_calls(chunk):
    """Five 512x768 images (24 patches each): chunk = 24 -> host chunks of one image, device sequences of 3 + 2;
    chunk = 48 -> host chunks of 2, 2, 1.  Results equal those of one chunk; repeated calls are identical."""
    codec, _, _ = make_codec("model_0", "fanin", compute="tensor")
    imgs = np.stack([O.synthetic_image(512, 768, 90 + i) for i in range(5)])
    cum = entry.cum_freq_table(_prob(codec, list(imgs), 128), 4096)
    want_cb, want_se, _ = codec.evaluate_images(imgs, 128, cum, out=np.zeros_like(imgs))
    want_rec = codec.roundtrip_images(imgs, 128, want_symbols=False)[0]
    codec.set_chunk_patches(chunk)
    d_imgs = torch.from_numpy(imgs).cuda()
    for _ in range(2):
        out = np.zeros_like(imgs)
        cb, se, _ = codec.evaluate_images(imgs, 128, cum, out=out)
        assert np.array_equal(cb, want_cb) and np.array_equal(se, want_se) and np.array_equal(out, want_rec)
        d_out = torch.zeros_like(d_imgs)
        cb, se, _ = codec.evaluate_images(d_imgs, 128, cum, out=d_out)
        assert cb.cpu().tolist() == want_cb.tolist() and se.cpu().tolist() == want_se.tolist()
        assert np.array_equal(d_out.cpu().numpy(), want_rec)
        cb, se, _ = codec.evaluate_images(d_imgs, 128, cum)
        assert cb.cpu().tolist() == want_cb.tolist() and se.cpu().tolist() == want_se.tolist()
    codec.check_status()
    codec.close()


def test_range_coder_runs_over_several_chunks():
    """128x128 images are one plain stream each.  3000 of them in five host chunks of 600: the range coder runs once
    2048 streams are pending (after the fourth chunk) and again for the last one; device buffers: two sequences."""
    codec, _, _ = make_codec("model_0", "fanin", compute="tensor")
    imgs = np.random.RandomState(5).randint(0, 256, size=(3000, 128, 128, 3), dtype=np.uint8)
    codec.hist_reset()
    sym = codec.encode_images(imgs, 128)
    counts = codec.hist_read().astype(np.float64)
    cum = entry.cum_freq_table(counts / counts.sum(), 4096)
    _, nbytes = codec.entropy_encode(sym, cum)
    d = imgs.astype(np.int64) - codec.decode_images(sym, 128, 128, 128)
    want_se = (d * d).sum(axis=(1, 2, 3))
    codec.set_chunk_patches(700)
    for src in (imgs, torch.from_numpy(imgs).cuda()):
        cb, se, _ = codec.evaluate_images(src, 128, cum)
        cb, se = (cb.cpu().numpy(), se.cpu().numpy()) if hasattr(cb, "cpu") else (cb, se)
        assert np.array_equal(cb, nbytes) and np.array_equal(se.astype(np.int64), want_se)
    codec.check_status()
    codec.close()


def test_histogram_accumulates_like_encode_images():
    codec, _, _ = make_codec("model_0", "fanin", compute="tensor")
    imgs = np.stack([O.synthetic_image(512, 768, 100 + i) for i in range(2)])
    codec.hist_reset()
    codec.evaluate_images(imgs, 128, [0, 2048, 4096])
    h_eval = codec.hist_read()
    codec.hist_reset()
    codec.encode_images(imgs, 128)
    assert np.array_equal(h_eval, codec.hist_read()) and h_eval.sum() > 0
    codec.close()


def test_errors():
    codec, _, _ = make_codec("model_0", "fanin", compute="tensor")
    imgs = np.stack([O.synthetic_image(256, 384, 110 + i) for i in range(2)])
    with pytest.raises(ValueError):
        codec.evaluate_images(imgs, 128, [1, 2048, 4096])      # table not starting at 0
    with pytest.raises(ValueError):
        codec.evaluate_images(imgs, 128, [0, 3000, 2048])      # decreasing entry
    with pytest.raises(ValueError):
        codec.evaluate_images(imgs, 128, [0, 0, 4096])         # symbol 0 has zero width: host buffers raise
    d_imgs = torch.from_numpy(imgs).cuda()
    codec.evaluate_images(d_imgs, 128, [0, 0, 4096])           # device buffers: asynchronous ...
    with pytest.raises(ValueError):
        codec.check_status()                                   # ... the error surfaces here
    codec.check_status()                                       # reported once
    with pytest.raises(ValueError):
        codec.evaluate_images(imgs, 128, [0, 2048, 4096], out=np.zeros((2, 256, 380, 3), np.uint8))
    with pytest.raises(ValueError):
        codec.evaluate_images(imgs, 128, [0, 2048, 4096], out=torch.zeros((2, 255, 384, 3), dtype=torch.uint8).cuda())
    cb, se, _ = codec.evaluate_images(np.zeros((0, 256, 384, 3), np.uint8), 128, [0, 2048, 4096])
    assert cb.shape == (0,) and se.shape == (0,)
    cb, se, _ = codec.evaluate_images(imgs, 128, [0, 2048, 4096])  # the handle still works
    assert (cb > 0).all()
    codec.close()
    # a handle with an encoder graph and no decoder graph
    enc, _ = params_for("model_0", "fanin")
    half = T.Codec.__new__(T.Codec)
    half.lib = L.load()
    half.device = 0
    half.quan_scale = 2
    h = C.c_void_p()
    assert half.lib.tic_create(C.byref(h), 0) == L.OK
    half._h = h
    half.enc_layers = T.variants.encoder_layers("model_0")
    half._set_graph(L.GRAPH_ENCODER, half.enc_layers, enc)
    half._check(half.lib.tic_set_norm(h, L.GRAPH_ENCODER, MEAN.ctypes.data, STD.ctypes.data))
    lut = T.inverse_sigmoid_lut(2)
    half._check(half.lib.tic_set_quantizer(h, 2, lut.ctypes.data))
    with pytest.raises(T.TicError):
        half.evaluate_images(imgs, 128, [0, 2048, 4096])
    half.close()
