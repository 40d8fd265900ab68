"""-m gpu parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Tolerances (BASELINE.json north_star): symbols bit-exact except at round-half boundaries
(mismatch rate <= 1e-5), reconstruction within 1e-3 max-abs on the 0..255 scale."""
import os

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
import tf_image_compression_b200 as T
from tf_image_compression_b200 import variants as V
from gpu_common import MEAN, STD, make_codec, params_for, patches_from_images, rel_err

pytestmark = pytest.mark.gpu

MODES = os.environ.get("TIC_TEST_MODES", "fp32,tensor").split(",")

# (variant, patch size, patches) — every BASELINE.json config plus the free table-driven variants
LAYER_CASES = [("model_0", 128, 3), ("model_1", 256, 1), ("base_model/input_256", 256, 1), ("base_model/ch_128", 128, 2),
               ("base_model/reduced_btn_32", 128, 2), ("model_3", 128, 2), ("model_2", 128, 2)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("variant,P,n", LAYER_CASES)
def test_layer_by_layer_activations(variant, P, n, mode):
    """Every intermediate activation of encoder and decoder (what sess.run on the op would fetch)."""
    codec, enc, dec = make_codec(variant, "fanin", compute=mode)
    rs = np.random.RandomState(7)
    x = rs.standard_normal((n, P, P, 3)).astype(np.float32)
    worst = []
    for graph, table, params, cin, x0 in (("encoder", O.VARIANTS[variant]["enc"], enc, 3, x), ("decoder", O.VARIANTS[variant]["dec"], dec, O.VARIANTS[variant]["bottleneck"], None)):
        if x0 is None:
            hb = codec.bottleneck_shape(P)[0]
            x0 = (rs.standard_normal((n, hb, hb, cin)) * 3).astype(np.float32)
        taps = []
        O.run_layers(x0, table, cin, params, taps=taps)
        prim = O.expand_layers(table, cin)
        for k, (scope, ref) in enumerate(taps, start=1):
            if prim[k - 1]["res_begin"]:
                continue  # cannot stop inside a residual block
            got = codec.run_layers(graph, x0, k)
            assert got.shape == ref.shape, (scope, got.shape, ref.shape)
            e = rel_err(got, ref)
            worst.append((e, graph, scope))
            assert e < 2e-5, f"{variant} {graph} layer {k} ({scope}): rel err {e:.3e}"
    print(f"[{variant}@{P} {mode}] worst layer rel err: {max(worst)}")
    codec.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("scheme", ["fanin", "reference"])
def test_model0_symbols_match_oracle(scheme, mode):
    """cfg1-shaped: model_0 @128; 96 patches = 393 216 symbols."""
    codec, enc, dec = make_codec("model_0", scheme, compute=mode)
    patches = patches_from_images(4, 512, 768, 128)  # 4 x 24 patches
    sym = codec.encode_patches(patches)
    ref = O.encoder(patches.astype(np.float32), "model_0", enc, MEAN, STD, 2)
    assert sym.shape == ref.shape == (96, 8, 8, 64) and sym.dtype == np.uint8
    mism = np.flatnonzero(sym.reshape(-1) != ref.reshape(-1))
    rate = mism.size / ref.size
    l64 = O.encoder_logits(patches.astype(np.float32), "model_0", enc, MEAN, STD, dtype=torch.float64).reshape(-1)
    scale = np.abs(l64).max()
    print(f"[model_0 {scheme} {mode}] mismatches {mism.size}/{ref.size} = {rate:.2e}; logit scale {scale:.3e}")
    # documented round-half boundary: a mismatch may only sit where the fp64 logit is within fp32
    # noise of the sigmoid == 0.5 threshold (dead zone (0, ~1.2e-7] plus accumulation error)
    if mism.size:
        assert np.abs(l64[mism]).max() < 1.5e-7 + 4e-6 * scale, np.abs(l64[mism]).max()
    if scheme == "fanin":
        assert rate <= 1e-5
    else:
        assert rate <= 5e-3  # 0.18 % of reference-init logits sit inside the dead zone (SURVEY.md §7.2)
    # f32 output (what sess.run returned) carries the same integers
    symf = codec.encode_patches(patches, out_dtype=np.float32)
    assert symf.dtype == np.float32 and np.array_equal(symf, sym.astype(np.float32))
    codec.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("variant,P,n", [("model_0", 128, 24), ("model_1", 256, 4), ("base_model/input_256", 256, 3),
                                         ("base_model/ch_128", 128, 6), ("base_model/ch_128", 256, 2),
                                         ("base_model/reduced_btn_32", 128, 8), ("model_3", 128, 6), ("model_2", 128, 6)])
def test_encode_decode_every_config(variant, P, n, mode):
    codec, enc, dec = make_codec(variant, "fanin", compute=mode)
    patches = patches_from_images(1, P, P * n, P, seed=11)
    assert patches.shape[0] == n
    sym = codec.encode_patches(patches)
    ref = O.encoder(patches.astype(np.float32), variant, enc, MEAN, STD, 2)
    nm = int((sym != ref).sum())
    assert sym.shape == ref.shape
    assert nm <= max(1, int(2e-5 * ref.size)), f"{variant}: {nm}/{ref.size} symbol mismatches"
    rec = codec.decode_patches(ref)
    rref = O.decoder(ref, variant, dec, MEAN, STD, 2)
    assert rec.shape == rref.shape == (n, P, P, 3)
    err = float(np.abs(rec - rref).max())
    print(f"[{variant}@{P} {mode}] symbol mismatches {nm}/{ref.size}; recon max-abs err {err:.3e}")
    assert err <= 1e-3
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_reference_init_reconstruction(mode):
    codec, enc, dec = make_codec("model_0", "reference", compute=mode)
    sym = np.random.RandomState(3).randint(0, 2, size=(24, 8, 8, 64)).astype(np.uint8)
    rec = codec.decode_patches(sym)
    rref = O.decoder(sym, "model_0", dec, MEAN, STD, 2)
    assert float(np.abs(rec - rref).max()) <= 1e-3
    codec.close()


def test_fused_crop_and_stitch_equal_the_host_helpers():
    """encode_images == encoder(crop_image_input_patches(...)); decode_images == around(concat_patches(decoder))."""
    codec, enc, dec = make_codec("model_0", "fanin")
    for (h, w) in [(512, 768), (300, 200), (129, 385)]:
        imgs = np.stack([O.synthetic_image(h, w, 20 + i) for i in range(3)])
        sym_i = codec.encode_images(imgs, 128)
        gh, gw = -(-h // 128), -(-w // 128)
        assert sym_i.shape == (3, gh * gw, 8, 8, 64)
        for i in range(3):
            patches = np.stack(T.utils.crop_image_input_patches(imgs[i], 128))
            assert np.array_equal(codec.encode_patches(patches), sym_i[i]), (h, w, i)
        rec_u8 = codec.decode_images(sym_i, h, w, 128)
        rec_f = codec.decode_images(sym_i, h, w, 128, out_dtype=np.float32)
        assert rec_u8.shape == (3, h, w, 3) and rec_u8.dtype == np.uint8
        for i in range(3):
            p = codec.decode_patches(sym_i[i])
            full = T.utils.concat_patches(list(p), h, w, 128)
            assert np.array_equal(full, rec_f[i])
            assert np.array_equal(np.around(full).astype(np.uint8), rec_u8[i])
        assert np.array_equal(codec.round_u8(rec_f), rec_u8)
    # oracle end to end on one image (encode.py:153-182 + decode.py:204-249 without the entropy coder)
    img = O.synthetic_image(300, 200, 99)
    s_ref, r_ref = O.codec_roundtrip(img, "model_0", enc, dec, MEAN, STD, 2, 128)
    s = codec.encode_images(img[None], 128)[0]
    assert (s != s_ref).sum() <= 1
    r = codec.decode_images(s_ref[None], 300, 200, 128)[0]
    assert np.abs(r.astype(int) - r_ref.astype(int)).max() <= 1 and (r != r_ref).mean() < 1e-4
    codec.close()


def test_histogram_and_position_sums_are_exact():
    codec, enc, dec = make_codec("base_model/reduced_btn_32", "fanin")
    patches = patches_from_images(2, 256, 384, 128, seed=5)
    codec.hist_reset()
    sym = codec.encode_patches(patches)
    counts = codec.hist_read()
    assert counts.dtype == np.uint64
    assert np.array_equal(counts, np.bincount(sym.reshape(-1), minlength=2))
    assert np.array_equal(counts.astype(np.float64), O.symbol_histogram(sym, 2))
    sym2 = codec.encode_patches(patches[:5])  # accumulates (get_encoded_distribution.py:126)
    assert np.array_equal(codec.hist_read(), counts + np.bincount(sym2.reshape(-1), minlength=2).astype(np.uint64))
    sums = codec.position_sums(sym)
    assert np.array_equal(sums, sym.reshape(sym.shape[0], -1).sum(0).astype(np.uint64))
    mean, _, _ = O.position_mean([sym])
    np.testing.assert_allclose(sums / sym.shape[0], mean, atol=1e-7)
    codec.close()


def test_quan_scale_256():
    codec, enc, dec = make_codec("model_0", "fanin", q=256)
    patches = patches_from_images(1, 256, 256, 128, seed=8)
    codec.hist_reset()
    sym = codec.encode_patches(patches)
    ref = O.encoder(patches.astype(np.float32), "model_0", enc, MEAN, STD, 256)
    d = np.abs(sym.astype(int) - ref.astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 1e-3
    assert np.array_equal(codec.hist_read(), np.bincount(sym.reshape(-1), minlength=256))
    rec = codec.decode_patches(ref)
    rref = O.decoder(ref, "model_0", dec, MEAN, STD, 256)
    assert float(np.abs(rec - rref).max()) <= 1e-3
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_postfilter_and_rmbe_match_oracle(mode):
    codec, enc, dec = make_codec("model_1", "fanin", compute=mode)
    pp = O.init_params(O.POSTFILTERS["rmbe"], 3, 77, "fanin")
    pm, ps = np.array([110.0, 108.0, 99.0], np.float32), np.array([55.0, 57.0, 60.0], np.float32)
    codec.set_postfilter(pp, pm, ps)
    tiles = patches_from_images(1, 128, 384, 128, seed=31).astype(np.float32)
    got = codec.postfilter_patches(tiles)
    ref = O.postfilter(tiles, "rmbe", pp, pm, ps)
    assert float(np.abs(got - ref).max()) <= 1e-3
    imgs = np.stack([O.synthetic_image(384, 448, 40 + i).astype(np.float32) for i in range(2)])
    want = np.stack([O.rmbe(im, lambda t: O.postfilter(t, "rmbe", pp, pm, ps)) for im in imgs])
    work = imgs.copy()
    codec.postfilter_images(work)
    assert float(np.abs(work - want).max()) <= 2e-3  # two chained passes
    # border strips are untouched (submit/2/rmbe/rmbe.py: first/last 64 px and remainders)
    assert np.array_equal(work[:, :64, :64], imgs[:, :64, :64])
    T.rmbe.bind(codec)
    single = T.rmbe.rmbe(imgs[0].copy())
    assert np.array_equal(single, work[0])
    # alternative 4-layer post-filter (rm_block_effect/model_1/model.py:107-168)
    pp1 = O.init_params(O.POSTFILTERS["rmbe_model_1"], 3, 78, "fanin")
    codec.set_postfilter(pp1, pm, ps, name="rmbe_model_1")
    got1 = codec.postfilter_patches(tiles[:2])
    ref1 = O.postfilter(tiles[:2], "rmbe_model_1", pp1, pm, ps)
    assert float(np.abs(got1 - ref1).max()) <= 1e-3
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_device_buffers_chunking_and_determinism(mode):
    codec, enc, dec = make_codec("model_0", "fanin", compute=mode)
    patches = patches_from_images(2, 384, 512, 128, seed=50)  # 24 patches
    base = codec.encode_patches(patches)
    d_in = torch.from_numpy(patches).cuda()
    d_out = codec.encode_patches(d_in)
    assert d_out.is_cuda and np.array_equal(d_out.cpu().numpy(), base)
    codec.set_chunk_patches(5)  # ragged chunks: 5,5,5,5,4
    assert np.array_equal(codec.encode_patches(patches), base)
    assert np.array_equal(codec.encode_patches(d_in).cpu().numpy(), base)
    rec = codec.decode_patches(base)
    codec.set_chunk_patches(7)
    assert np.array_equal(codec.decode_patches(base), rec)
    assert np.array_equal(codec.decode_patches(torch.from_numpy(base).cuda()).cpu().numpy(), rec)
    # f32 patches give the same symbols as u8 patches (normalisation LUT == arithmetic)
    assert np.array_equal(codec.encode_patches(patches.astype(np.float32)), base)
    assert codec.launch_count > 0 and codec.last_kernel_ms() > 0
    # empty batch
    assert codec.encode_patches(np.zeros((0, 128, 128, 3), np.uint8)).shape == (0, 8, 8, 64)
    codec.close()


def test_reference_module_surface_and_errors():
    codec, enc, dec = make_codec("model_0", "fanin")
    model = T.ModelModule("model_0", codec)
    patches = patches_from_images(1, 128, 256, 128, seed=60)
    out = model.encoder(patches.astype(np.float32), 128, 2)  # float32 feed like encode.py:140,157
    assert out.dtype == np.float32 and out.shape == (2, 8, 8, 64) and set(np.unique(out)) <= {0.0, 1.0}
    seq = np.asarray(out).reshape(-1).astype(int).tolist()  # encode.py:175-182
    assert len(seq) == 2 * 8 * 8 * 64
    rec = model.decoder(out, 2)
    assert rec.shape == (2, 128, 128, 3) and rec.min() >= 0 and rec.max() <= 255
    with pytest.raises(ValueError):
        model.decoder(out + 0.5, 2)
    with pytest.raises(ValueError):
        model.encoder(patches, 128, 3)
    with pytest.raises(ValueError):
        codec.encode_patches(np.zeros((2, 128, 64, 3), np.uint8))
    with pytest.raises(ValueError):
        codec.decode_patches(np.zeros((2, 8, 8, 32), np.uint8))
    with pytest.raises(T.TicError):
        codec.postfilter_patches(np.zeros((1, 128, 128, 3), np.float32))
    with pytest.raises(KeyError):
        T.Codec("model_0", enc_params={"encode_0/kernel": np.zeros((3, 3, 3, 32), np.float32)})
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_golden_fixture_cfg1(mode):
    """BASELINE config 1 (768x512 image, model_0, 128x128 patches) against the committed fixture
    (tests/golden/make_golden.py)."""
    import hashlib
    from pathlib import Path
    z = np.load(Path(__file__).parent / "golden" / "cfg1_model0_768x512.npz")
    image = O.synthetic_image(512, 768, 1234)
    assert hashlib.sha256(image.tobytes()).hexdigest() == str(z["image_sha256"])
    ov = O.VARIANTS["model_0"]
    enc = O.init_params(ov["enc"], 3, 1234, "fanin")
    dec = O.init_params(ov["dec"], ov["bottleneck"], 1235, "fanin")
    dec = O.condition_decoder("model_0", dec, 2)
    chk = [float(sum(np.float64(v).sum() for v in enc.values())), float(sum(np.float64(v).sum() for v in dec.values()))]
    np.testing.assert_allclose(chk, z["weight_checksum"], rtol=0, atol=1e-9)
    codec = T.Codec("model_0", quan_scale=2, mean=z["mean"], std=z["std"], enc_params=enc, dec_params=dec, compute=mode)
    sym = codec.encode_images(image[None], 128)[0]
    assert sym.shape == (24, 8, 8, 64)
    packed = np.packbits(sym.reshape(-1))
    assert (np.unpackbits(packed ^ z["symbols_packed"]).sum()) <= 1
    rec = codec.decode_images(np.unpackbits(z["symbols_packed"]).reshape(1, 24, 8, 8, 64), 512, 768, 128)[0]
    mask = np.unpackbits(z["recon_mask_packed"], count=rec.size).astype(bool)
    d = np.abs(rec.reshape(-1)[mask].astype(int) - z["recon_sample"].astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 1e-4
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_full_size_properties_cfg2_shard(mode):
    """BASELINE config 2 at one GPU's 8-image share (8 x 2048x1536, 1 536 patches): size-independent
    properties — determinism, batch == per-image, histogram == symbol count, decode idempotence."""
    codec, enc, dec = make_codec("model_0", "fanin", compute=mode)
    rs = np.random.RandomState(1234)
    imgs = rs.randint(0, 256, size=(8, 1536, 2048, 3), dtype=np.uint8)
    d_imgs = torch.from_numpy(imgs).cuda()
    codec.hist_reset()
    sym = codec.encode_images(d_imgs, 128)
    assert tuple(sym.shape) == (8, 192, 8, 8, 64)
    counts = codec.hist_read()
    assert int(counts.sum()) == sym.numel() and int(counts[1]) == int(sym.sum())
    assert torch.equal(codec.encode_images(d_imgs, 128), sym)  # deterministic
    one = codec.encode_images(d_imgs[5:6].contiguous(), 128)
    assert torch.equal(one[0], sym[5])  # batch == per image
    host = codec.encode_images(imgs[:2], 128)  # host path == device path
    assert np.array_equal(host, sym[:2].cpu().numpy())
    rec = codec.decode_images(sym, 1536, 2048, 128)
    assert tuple(rec.shape) == (8, 1536, 2048, 3) and rec.dtype == torch.uint8
    assert torch.equal(codec.decode_images(sym, 1536, 2048, 128), rec)
    # spot-check one patch of one image against the oracle
    p = imgs[3, 128:256, 256:384][None].astype(np.float32)
    assert (O.encoder(p, "model_0", enc, MEAN, STD, 2)[0] != sym[3, 1 * 16 + 2].cpu().numpy()).sum() <= 1
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_cfg4_distribution_table_and_bitstreams(mode, tmp_path):
    """BASELINE config 4: base_model/reduced_btn_32 (bottleneck_channel from config), dataset-wide symbol table
    (fused histogram == np.histogram of the oracle's symbols, get_encoded_distribution.py:113-134), range-coded
    files byte-identical to coding the oracle's symbols, and the decode side of the round trip."""
    from tf_image_compression_b200 import entry, range_coder
    variant = "base_model/reduced_btn_32"
    codec, enc, dec = make_codec(variant, "fanin", compute=mode)
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=128, bottleneck_channel=32)
    images = [O.synthetic_image(256, 384, 70 + i) for i in range(3)] + [O.synthetic_image(200, 300, 90)]  # ragged size too
    names = [f"/data/x/img_{i}.png" for i in range(len(images))]
    patches = np.stack([p for im in images for p in O.crop_image_input_patches(im, 128)])
    prob = entry.get_distribution(codec, patches)
    counts = codec.hist_read()
    ref_sym = O.encoder(patches.astype(np.float32), variant, enc, MEAN, STD, 2).astype(np.uint8)
    gpu_sym = codec.encode_patches(patches)
    mism = int((gpu_sym != ref_sym).sum())
    assert mism <= max(1, int(1e-5 * ref_sym.size)), mism  # round-half boundary only (north_star: <= 1e-5)
    # the fused histogram is exactly np.histogram of the emitted symbols (get_encoded_distribution.py:121-126)
    assert np.array_equal(counts.astype(np.int64), np.histogram(gpu_sym, bins=[0, 1, 2])[0])
    assert np.allclose(prob, counts / counts.sum())
    out = entry.compress(codec, images, names, cfg, prob, str(tmp_path / "enc"))
    cum = entry.cum_freq_table(prob, 4096)
    k = 0
    for (path, nbytes), im in zip(out, images):
        npatch = len(O.crop_image_input_patches(im, 128))
        stem, eshape, n, h, w = entry.parse_encoded_name(os.path.basename(path), cfg)
        assert eshape == (32, 32, 32) and n == npatch * 32 * 32 * 32 and (h, w) == im.shape[:2]
        # bitstreams are byte-identical wherever the symbols are identical: code the oracle's symbols with the same table
        if np.array_equal(gpu_sym[k:k + npatch], ref_sym[k:k + npatch]):
            ref_path = tmp_path / "ref.bin"
            e = range_coder.RangeEncoder(str(ref_path))
            e.encode(ref_sym[k:k + npatch].reshape(-1), cum)
            e.close()
            assert ref_path.read_bytes() == open(path, "rb").read()
        assert nbytes == os.path.getsize(path)
        k += npatch
    # bpp delta (BASELINE metric): the oracle's symbols through the same coder and table
    ref_bytes, k = [], 0
    for im in images:
        npatch = len(O.crop_image_input_patches(im, 128))
        e = range_coder.RangeEncoder(str(tmp_path / "ref_bpp.bin"))
        e.encode(ref_sym[k:k + npatch].reshape(-1), cum)
        e.close()
        ref_bytes.append(os.path.getsize(tmp_path / "ref_bpp.bin"))
        k += npatch
    bpp_gpu, bpp_ref = entry.bpp([b for _, b in out], images), entry.bpp(ref_bytes, images)
    assert abs(bpp_gpu - bpp_ref) <= 1e-4 * bpp_ref, (bpp_gpu, bpp_ref)
    oracle_sym = ref_sym
    ref_sym = gpu_sym  # the decode side is checked on the symbols that were actually coded
    rec = entry.uncompress(codec, str(tmp_path / "enc"), cfg, prob)
    assert sorted(rec) == [f"img_{i}" for i in range(len(images))]
    k = 0
    for i, im in enumerate(images):
        npatch = len(O.crop_image_input_patches(im, 128))
        want = O.around_u8(O.concat_patches(list(O.decoder(ref_sym[k:k + npatch], variant, dec, MEAN, STD, 2)), im.shape[0], im.shape[1], 128))
        d = np.abs(rec[f"img_{i}"].astype(int) - want.astype(int))
        assert rec[f"img_{i}"].shape == im.shape and d.max() <= 1 and (d != 0).mean() < 1e-4
        k += npatch
    # PSNR delta (BASELINE metric, north_star: within 0.01 dB): the oracle's own round trip (its symbols, its decoder)
    wants, k = [], 0
    for im in images:
        npatch = len(O.crop_image_input_patches(im, 128))
        wants.append(O.around_u8(O.concat_patches(list(O.decoder(oracle_sym[k:k + npatch], variant, dec, MEAN, STD, 2)),
                                                  im.shape[0], im.shape[1], 128)))
        k += npatch
    psnr_gpu = entry.psnr(images, [rec[f"img_{i}"] for i in range(len(images))])
    psnr_ref = entry.psnr(images, wants)
    assert np.isfinite(psnr_gpu) and abs(psnr_gpu - psnr_ref) <= 0.01, (psnr_gpu, psnr_ref)
    assert bpp_gpu > 0
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_cfg5_model1_decode_and_rmbe(mode):
    """BASELINE config 5: model_1 (P = 256) decode -> stitch -> rmbe post-filter -> round, call order of
    submit/2/decoder.py:183-198; oracle parity on a 512x768 image, size-independent properties at 2048x1536."""
    codec, enc, dec = make_codec("model_1", "fanin", compute=mode)
    pp = O.init_params(O.POSTFILTERS["rmbe"], 3, 77, "fanin")
    pm, ps = np.array([110.0, 108.0, 99.0], np.float32), np.array([55.0, 57.0, 60.0], np.float32)
    codec.set_postfilter(pp, pm, ps)
    rs = np.random.RandomState(8)
    sym = rs.randint(0, 2, size=(1, 6, 16, 16, 64)).astype(np.uint8)  # 512x768 at P = 256: 2 x 3 patches
    got = codec.decode_images(sym, 512, 768, 256, out_dtype=np.float32)
    want = O.concat_patches(list(O.decoder(sym[0], "model_1", dec, MEAN, STD, 2)), 512, 768, 256)
    assert float(np.abs(got[0] - want).max()) <= 1e-3
    codec.postfilter_images(got)
    want = O.rmbe(want.astype(np.float32), lambda t: O.postfilter(t, "rmbe", pp, pm, ps))
    assert float(np.abs(got[0] - want).max()) <= 3e-3  # decoder + two chained filter passes
    out8 = codec.round_u8(got)
    assert out8.dtype == np.uint8 and np.abs(out8[0].astype(int) - O.around_u8(want).astype(int)).max() <= 1
    # full size: 2048x1536 -> 48 patches of 256, 356 filter tiles per image; deterministic, borders untouched
    big = torch.from_numpy(rs.randint(0, 2, size=(2, 48, 16, 16, 64)).astype(np.uint8)).cuda()
    img = codec.decode_images(big, 1536, 2048, 256, out_dtype=np.float32)
    before = img.clone()
    codec.postfilter_images(img)
    again = before.clone()
    codec.postfilter_images(again)
    assert torch.equal(img, again)
    assert torch.equal(img[:, :64, :64], before[:, :64, :64]) and not torch.equal(img[:, 64:192, 64:192], before[:, 64:192, 64:192])
    assert float(img.min()) >= 0.0 and float(img.max()) <= 255.0
    codec.close()


@pytest.mark.parametrize("mode", MODES)
def test_roundtrip_equals_encode_then_decode(mode):
    """tic_roundtrip_images (test.py:95-146, encoder and decoder in one graph) == tic_encode_images followed by
    tic_decode_images, bit for bit: host buffers (streamed, several chunks, pinned and pageable), device buffers (one
    launch sequence and two),
    images that need reflect padding, float output, no symbol read-back; the histogram counts every symbol once."""
    codec, enc, dec = make_codec("model_0", "fanin", compute=mode)
    rs = np.random.RandomState(77)
    imgs = rs.randint(0, 256, size=(5, 300, 410, 3), dtype=np.uint8)  # 3 x 4 patches per image, padded bottom / right
    sym = codec.encode_images(imgs, 128)
    rec = codec.decode_images(sym, 300, 410, 128)
    codec.set_chunk_patches(24)  # host: 2 images per chunk -> 3 chunks, the last one ragged
    codec.hist_reset()
    r2, s2 = codec.roundtrip_images(imgs, 128)
    assert np.array_equal(s2, sym) and np.array_equal(r2, rec)
    assert int(codec.hist_read().sum()) == sym.size
    pinned = torch.from_numpy(imgs).pin_memory()
    out_p = torch.empty((5, 300, 410, 3), dtype=torch.uint8).pin_memory()
    r3, s3 = codec.roundtrip_images(pinned, 128, out=out_p, want_symbols=False)
    assert s3 is None and np.array_equal(r3.numpy(), rec)
    rf, _ = codec.roundtrip_images(imgs, 128, out_dtype=np.float32)
    assert np.array_equal(rf, codec.decode_images(sym, 300, 410, 128, out_dtype=np.float32))
    rd, sd = codec.roundtrip_images(torch.from_numpy(imgs).cuda(), 128)
    assert rd.is_cuda and np.array_equal(sd.cpu().numpy(), sym) and np.array_equal(rd.cpu().numpy(), rec)
    # the oracle's round trip of one image (crop -> encoder -> decoder -> stitch -> np.around)
    o = O.codec_roundtrip(imgs[1], "model_0", enc, dec, MEAN, STD, 2, 128)
    o_img = o[1] if isinstance(o, tuple) else o
    assert np.abs(o_img.astype(np.int32) - rec[1].astype(np.int32)).max() <= 1
    from tf_image_compression_b200 import entry
    outs = entry.compress_and_uncompress(codec, [imgs[0], imgs[1][:200, :256].copy(), imgs[2]], {"patch_size": 128})
    assert np.array_equal(outs[0], rec[0]) and np.array_equal(outs[2], rec[2]) and outs[1].shape == (200, 256, 3)
    # device buffers over two launch sequences (one image per chunk: 3 + 2 images), encoder then decoder per sequence
    codec.set_chunk_patches(12)
    rd, sd = codec.roundtrip_images(torch.from_numpy(imgs).cuda(), 128)
    assert np.array_equal(sd.cpu().numpy(), sym) and np.array_equal(rd.cpu().numpy(), rec)
    codec.close()


def test_restore_params_from_tf_v2_checkpoint(tmp_path):
    """utils.restore_params (utils/utils.py:84-93): model_N/params_for_test/params written in the TF-V2 bundle layout
    -> checkpoint.restore_params -> the same symbols and reconstruction as the codec given the arrays directly."""
    from tf_image_compression_b200 import checkpoint as K
    codec, enc, dec = make_codec("model_0", "fanin", compute="tensor")
    patches = patches_from_images(1, 256, 256, 128, seed=3)
    sym = codec.encode_patches(patches)
    rec = codec.decode_patches(sym)
    codec.close()
    K.write_checkpoint(tmp_path / "model_0" / "params_for_test" / "params", {**enc, **dec})
    fresh = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, compute="tensor", seed=5)  # reference-init weights
    assert not np.array_equal(fresh.encode_patches(patches), sym)
    K.restore_params(fresh, model_num=0, root=str(tmp_path))
    assert np.array_equal(fresh.encode_patches(patches), sym)
    assert np.array_equal(fresh.decode_patches(sym), rec)
    with pytest.raises(FileNotFoundError):
        K.restore_params(fresh, params_file=str(tmp_path / "absent" / "params"))
    fresh.close()


def test_nccl_table_allreduce():
    """The path's one collective on real GPUs (needs two): tests/nccl_table_check.py under torchrun."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gpurun --gpus 2); the gloo world-size-2 test covers the host logic on CPU")
    script = os.path.join(os.path.dirname(__file__), "nccl_table_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", script], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "nccl table check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_full_size_roundtrip_host_equals_device():
    """BASELINE config 2 at a quarter of one GPU's share (16 x 2048x1536, 3072 patches): the streamed host-to-host round
    trip (16 chunks, both PCIe directions busy) is bit-identical to the device-resident calls, twice in a row."""
    codec, enc, dec = make_codec("model_0", "fanin", compute="tensor")
    rs = np.random.RandomState(4321)
    imgs = torch.from_numpy(rs.randint(0, 256, size=(16, 1536, 2048, 3), dtype=np.uint8)).pin_memory()
    d_imgs = imgs.cuda()
    sym = codec.encode_images(d_imgs, 128)
    rec = codec.decode_images(sym, 1536, 2048, 128)
    out = torch.empty((16, 1536, 2048, 3), dtype=torch.uint8).pin_memory()
    osym = torch.empty(tuple(sym.shape), dtype=torch.uint8).pin_memory()
    for _ in range(2):
        out.zero_()
        codec.roundtrip_images(imgs, 128, out=out, out_symbols=osym)
        assert torch.equal(osym, sym.cpu()) and torch.equal(out, rec.cpu())
    # error of the codec itself is irrelevant here (random-free fan-in weights); the crop -> stitch geometry is not:
    assert tuple(out.shape) == tuple(imgs.shape)
    codec.close()
