"""-m gpu parity tests, round 2: realistic dynamic range, the TF32 compute modes, the fp16-range guard, the
cal_encoded_distribution outputs, the GPU entropy stage (byte identity with the host coder), stream / device handling
of the C ABI, and the reference's unmodified entry points over the real Codec (where a reference checkout exists)."""
import os
import time
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import codec_oracle as O
import tf_image_compression_b200 as T
from tf_image_compression_b200 import entry, range_coder
from gpu_common import MEAN, STD, make_codec, params_for, patches_from_images

pytestmark = pytest.mark.gpu


# ---- decoder parity at realistic dynamic range (VERDICT r1, weak #3) ----------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tensor"])
@pytest.mark.parametrize("variant", ["model_0", "model_1", "model_3", "model_2"])
def test_decoder_parity_at_realistic_range(variant, mode):
    """A trained decoder's pre-denormalisation output has std ~ 1 (the data is normalised to unit variance,
    model_0/model.py:44,251) and the 0..255 clip is active.  condition_decoder(target_std=1.0) gives a random decoder
    that range; P = 256 (the reference's config.json patch size) for model_0 / model_1, P = 128 for the submitted codecs
    model_3 (submit/2, submit/3) and model_2 (submit/1).  The fp64 evaluation of the same graph is the arbiter: the GPU
    result must be as close to it as the fp32 oracle is, and within the north-star bound of the fp32 oracle.  The fp16
    range guard of the tensor path must not trip at this range."""
    P = 128 if variant in ("model_3", "model_2") else 256
    ov = O.VARIANTS[variant]
    dec = O.condition_decoder(variant, O.init_params(ov["dec"], ov["bottleneck"], 1235, "fanin"), 2, target_std=1.0)
    enc = O.init_params(ov["enc"], 3, 1234, "fanin")
    codec = T.Codec(variant, quan_scale=2, mean=MEAN, std=STD, enc_params=enc, dec_params=dec, compute=mode)
    sym = np.random.RandomState(21).randint(0, 2, size=(3, *codec.bottleneck_shape(P))).astype(np.uint8)
    got = codec.decode_patches(sym)
    codec.check_status()
    ref32 = O.decoder(sym, variant, dec, MEAN, STD, 2)
    ref64 = O.decoder(sym, variant, dec, MEAN, STD, 2, dtype=torch.float64)
    clipped = float(((ref64 <= 0.0) | (ref64 >= 255.0)).mean())
    e_gpu64, e_ref64, e_gpu32 = (float(np.abs(got - ref64).max()), float(np.abs(ref32 - ref64).max()),
                                 float(np.abs(got - ref32).max()))
    print(f"[{variant}@{P} {mode}] clipped {clipped:.3f}; |gpu-f64| {e_gpu64:.3e}  |oracle32-f64| {e_ref64:.3e}  |gpu-oracle32| {e_gpu32:.3e}")
    assert got.shape == (3, P, P, 3)
    assert 0.005 < clipped < 0.5, clipped        # clipping is active but the image is not saturated
    assert float(np.std(ref64)) > 40.0           # realistic spread on the 0..255 scale
    assert e_gpu32 <= 1e-3                       # north_star: reconstruction within 1e-3 max-abs of the fp32 reference
    assert e_gpu64 <= 1e-3 and e_gpu64 <= 4.0 * e_ref64 + 2e-4
    # rounded images: np.around of two float images that differ by < 1e-3 may differ by one grey level at .5 boundaries
    d = np.abs(np.around(got).astype(int) - np.around(ref32).astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 1e-3
    codec.close()


# ---- fused layer pairs (tic_fused_enc16.cuh / tic_fused16.cuh) on the shapes that stress their tiling ----------------
@pytest.mark.parametrize("variant,P,h,w,nimg", [("model_0", 64, 64, 192, 1),       # one tile row per patch, 3 patches (odd)
                                                ("model_0", 128, 128, 384, 3),     # 9 patches: pairs straddle images, odd tail
                                                ("model_0", 256, 256, 512, 1),     # eight tile columns (the maximum)
                                                ("base_model/input_256", 256, 256, 256, 3),
                                                ("model_1", 128, 256, 128, 1)])
def test_fused_layer_pairs_on_edge_shapes(variant, P, h, w, nimg):
    """compute = tensor, u8 images whose patch grid covers them exactly: the first two encoder layers and the last two
    decoder layers run as the back-to-back kernels.  A CTA pair walks two patches in lock-step, so odd patch counts leave
    a pair with one patch beyond the batch; P = 64 has a single tile row (no halo row from below / above), P = 256 the
    maximum number of tile columns.  Symbols and reconstruction against the oracle, and against the fp32 CUDA-core path."""
    codec, enc, dec = make_codec(variant, "fanin", compute="tensor")
    imgs = np.stack([O.synthetic_image(h, w, 40 + i) for i in range(nimg)])
    patches = np.stack([pt for im in imgs for pt in O.crop_image_input_patches(im, P)])
    sym = codec.encode_images(imgs, P)
    ref = O.encoder(patches.astype(np.float32), variant, enc, MEAN, STD, 2)
    got = sym.reshape(ref.shape)
    nm = int((got != ref).sum())
    assert nm <= max(1, int(2e-5 * ref.size)), f"{variant}@{P}: {nm}/{ref.size} symbol mismatches"
    rec = codec.decode_images(ref.reshape(sym.shape), h, w, P, out_dtype=np.float32)
    rref = O.decoder(ref, variant, dec, MEAN, STD, 2)
    per = patches.shape[0] // nimg
    for i in range(nimg):
        full = T.utils.concat_patches(list(rref[i * per:(i + 1) * per]), h, w, P)
        err = float(np.abs(rec[i] - full).max())
        assert err <= 1e-3, (variant, P, i, err)
    rec_u8 = codec.decode_images(ref.reshape(sym.shape), h, w, P)
    assert np.abs(rec_u8.astype(int) - np.around(rec).astype(int)).max() == 0
    # the same calls on the CUDA-core fp32 path (no fused kernels)
    codec.set_compute("fp32")
    sym32 = codec.encode_images(imgs, P)
    assert int((sym32 != sym).sum()) <= max(1, int(2e-5 * ref.size))
    rec32 = codec.decode_images(ref.reshape(sym.shape), h, w, P, out_dtype=np.float32)
    assert float(np.abs(rec32 - rec).max()) <= 1e-3
    print(f"[fused pairs {variant}@{P} {nimg}x{h}x{w}] symbol mismatches {nm}/{ref.size}")
    codec.close()


def test_tensor_path_launch_counts_guard_against_silent_fallbacks():
    """model_0 at P = 128 on exact-grid u8 images, compute = tensor: 8 encoder launches (the fused first pair, encode_2,
    encode_3 in ONE launch, four residual-block convs, encode_4) and 10 decoder launches (symbols -> pair planes, decode_4,
    four convs, decode_3 as two phase-stacked slices, decode_2, the fused last pair).  A layer that silently dropped to
    an un-fused or sliced plan shows up here before it shows up in the bench."""
    codec, enc, dec = make_codec("model_0", "fanin", compute="tensor")
    imgs = torch.from_numpy(np.stack([O.synthetic_image(256, 384, 80 + i) for i in range(4)])).cuda()
    sym = codec.encode_images(imgs, 128)            # first call: lazily built weight images add launches
    rec = codec.decode_images(sym, 256, 384, 128)
    n0 = codec.launch_count
    codec.encode_images(imgs, 128)
    n1 = codec.launch_count
    codec.decode_images(sym, 256, 384, 128)
    n2 = codec.launch_count
    assert (n1 - n0, n2 - n1) == (8, 10), (n1 - n0, n2 - n1)
    assert tuple(rec.shape) == (4, 256, 384, 3)
    codec.close()


def test_fused_encoder_with_unusual_normalisation_constants():
    """The fused encoder folds 1 / std into the first layer's weights and works on the exact integers x - round(mean)
    (tic_fused_enc16.cuh, FusedEncNorm): identity normalisation, a mean of 0.5 (rounds to even), a tiny and a huge std, and
    a change of the constants on a live handle (tic_set_norm) must all agree with the oracle and the fp32 path."""
    enc, dec = params_for("model_0", "fanin")
    imgs = np.stack([O.synthetic_image(128, 256, 60 + i) for i in range(2)])
    patches = np.stack([pt for im in imgs for pt in O.crop_image_input_patches(im, 128)])
    codec = None
    for mean, std in ((np.zeros(3, np.float32), np.ones(3, np.float32)),
                      (np.array([0.5, 200.7, 33.3], np.float32), np.array([1.0, 255.0, 0.37], np.float32)),
                      (MEAN, STD)):
        if codec is None:
            codec = T.Codec("model_0", quan_scale=2, mean=mean, std=std, enc_params=enc, dec_params=dec, compute="tensor")
        else:   # same handle, new constants: the cached first-layer operand image must be rebuilt
            codec.mean, codec.std = np.ascontiguousarray(mean, np.float32), np.ascontiguousarray(std, np.float32)
            for g in (T._lib.GRAPH_ENCODER, T._lib.GRAPH_DECODER):
                codec._check(codec.lib.tic_set_norm(codec._h, g, codec.mean.ctypes.data, codec.std.ctypes.data))
        codec.set_compute("tensor")
        sym = codec.encode_images(imgs, 128)
        ref = O.encoder(patches.astype(np.float32), "model_0", enc, mean, std, 2)
        nm = int((sym.reshape(ref.shape) != ref).sum())
        codec.set_compute("fp32")
        nm32 = int((codec.encode_images(imgs, 128) != sym).sum())
        print(f"[fused encoder, mean {mean.tolist()} std {std.tolist()}] mismatches vs oracle {nm}/{ref.size}, vs fp32 path {nm32}")
        assert nm <= max(1, int(2e-5 * ref.size)) and nm32 <= max(1, int(2e-5 * ref.size))
    codec.close()


# ---- the first tensor path: 3xTF32 (error-compensated) and single-pass TF32 (VERDICT r1, weak #4) ----------------
def test_tf32_compute_modes():
    """TIC_COMPUTE_TENSOR_3XTF32 meets the same bars as the fp32 path; TIC_COMPUTE_TENSOR_TF32 is the documented fast
    mode: single-pass TF32 operands (10-bit significand) flip ~1e-4 of the binary symbols (SURVEY.md §7: 1.4e-4 - 1.7e-4
    in simulation) and is NOT parity-grade — the test states its measured rate and bounds it."""
    enc, dec = params_for("model_0", "fanin")
    patches = patches_from_images(4, 512, 768, 128)  # 96 patches, 393 216 symbols
    ref = O.encoder(patches.astype(np.float32), "model_0", enc, MEAN, STD, 2)
    sym_dec = np.random.RandomState(3).randint(0, 2, size=(24, 8, 8, 64)).astype(np.uint8)
    rref = O.decoder(sym_dec, "model_0", dec, MEAN, STD, 2)
    rates = {}
    for mode in ("3xtf32", "tf32"):
        codec = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, enc_params=enc, dec_params=dec, compute=mode)
        sym = codec.encode_patches(patches)
        rate = float((sym != ref).mean())
        err = float(np.abs(codec.decode_patches(sym_dec) - rref).max())
        rates[mode] = (rate, err)
        print(f"[model_0 {mode}] symbol mismatch rate {rate:.3e} ({int((sym != ref).sum())}/{ref.size}); recon max-abs err {err:.3e}")
        codec.close()
    # measured on B200 (round 2): 3xtf32 0 / 393 216 mismatches, recon 7.6e-4;  tf32 86 / 393 216 = 2.2e-4, recon 0.49 grey levels
    assert rates["3xtf32"][0] <= 1e-5 and rates["3xtf32"][1] <= 1e-3
    assert rates["tf32"][0] <= 1e-3 and rates["tf32"][1] <= 2.0  # fast mode: outside the north-star bars, as documented
    assert rates["tf32"][0] >= rates["3xtf32"][0]


# ---- fp16-range guard (VERDICT r1, weak #6) ----------------------------------------------------------------------
def test_fp16_range_guard():
    """TIC_COMPUTE_TENSOR_F16X3 keeps activations as fp16 pairs: |x| >= 65504 cannot be represented.  Every kernel that
    writes pair planes checks; the handle turns sticky-invalid (TIC_ERR_UNSUPPORTED) instead of returning garbage, the
    fp32 path computes the same graph fine, and switching modes clears the flag."""
    enc, dec = params_for("model_0", "fanin")
    big = dict(enc)
    big["encode_1/kernel"] = (enc["encode_1/kernel"] * np.float32(3.0e4)).astype(np.float32)  # encode_1 output ~1e5
    patches = patches_from_images(1, 128, 256, 128, seed=9)
    codec = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, enc_params=big, dec_params=dec, compute="tensor")
    with pytest.raises(T.TicError, match="fp16 range"):
        codec.encode_patches(patches)
    with pytest.raises(T.TicError, match="fp16 range"):  # sticky: later calls fail too
        codec.encode_patches(patches)
    with pytest.raises(T.TicError, match="fp16 range"):
        codec.check_status()
    codec.set_compute("fp32")  # clears the flag; the exact path has no such limit
    s32 = codec.encode_patches(patches)
    ref = O.encoder(patches.astype(np.float32), "model_0", big, MEAN, STD, 2)
    assert (s32 != ref).mean() <= 1e-3  # huge logits: sigmoid saturates, only boundary cases can differ
    codec.check_status()
    # device-buffer calls are asynchronous: the status surfaces through check_status()
    codec.set_compute("tensor")
    d_in = torch.from_numpy(patches).cuda()
    codec.encode_patches(d_in)
    with pytest.raises(T.TicError, match="fp16 range"):
        codec.check_status()
    codec.close()
    # in-range weights never trip it
    ok = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, enc_params=enc, dec_params=dec, compute="tensor")
    ok.encode_patches(patches)
    ok.check_status()
    ok.close()


# ---- cal_encoded_distribution outputs (VERDICT r1, missing #5) ----------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tensor"])
def test_cal_distribution_outputs(mode):
    """prob = [1 - mean(seq_prob), mean(seq_prob)] and encoded_order (cal_encoded_distribution.py:111-149) from exact
    per-batch device sums == the oracle's literal restatement fed with the same symbols in batches of 64."""
    codec, enc, dec = make_codec("base_model/reduced_btn_32", "fanin", compute=mode)
    patches = patches_from_images(25, 256, 384, 128, seed=15)  # 150 patches: batches of 64, 64, 22
    prob, order, seq_prob = entry.cal_distribution(codec, patches)
    sym = codec.encode_patches(patches)
    batches = [sym[i:i + 64].astype(np.float32) for i in range(0, len(sym), 64)]
    o_seq, o_prob, o_order = O.position_mean(batches)
    assert np.array_equal(seq_prob, o_seq) and np.array_equal(prob, o_prob) and order == o_order
    assert len(order) == 32 * 32 * 32 and sorted(order) == list(range(len(order)))
    assert abs(prob.sum() - 1.0) < 1e-12 and abs(prob[1] - sym.mean()) < 1e-6
    sums = codec.position_sums_batched(torch.from_numpy(sym).cuda(), 64).cpu().numpy()
    assert sums.shape == (3, 32 * 32 * 32)
    assert np.array_equal(sums, np.stack([b.reshape(len(b), -1).sum(0) for b in batches]).astype(np.int64))
    codec.close()


# ---- GPU entropy stage (SURVEY §8 f4) -----------------------------------------------------------------------------
def _host_streams(sym2d, cum):
    return range_coder.encode_streams(sym2d, cum, threads=0)


@pytest.mark.parametrize("case", ["binary_pow2", "binary_skewed", "binary_total_3000", "q16", "q256_unaligned", "segmented_ragged",
                                  "segmented_q16"])
def test_entropy_stage_is_byte_identical_to_the_host_coder(case):
    codec, _, _ = make_codec("model_0", "fanin")
    rs = np.random.RandomState({"binary_pow2": 1, "binary_skewed": 2, "binary_total_3000": 3, "q16": 4, "q256_unaligned": 5,
                                "segmented_ragged": 6, "segmented_q16": 7}[case])
    if case == "binary_pow2":
        sym = (rs.rand(7, 24576) < 0.45).astype(np.uint8)
        cum = entry.cum_freq_table(np.bincount(sym.reshape(-1), minlength=2) / sym.size, 4096)
    elif case == "binary_skewed":  # long runs of the likely symbol: carries through 0xFF runs
        sym = (rs.rand(5, 65536) < 0.001).astype(np.uint8)
        cum = [0, 4095, 4096]
    elif case == "binary_total_3000":  # not a power of two: the division path
        sym = (rs.rand(3, 4096) < 0.3).astype(np.uint8)
        cum = [0, 2100, 3000]
    elif case == "q16":
        p = rs.dirichlet([0.5] * 16)
        sym = rs.choice(16, size=(4, 8192), p=p).astype(np.uint8)
        cum = range_coder.prob_to_cum_freq(p, resolution=1024)
    elif case == "segmented_ragged":  # container format (include/tic_rc_core.h); odd length: unaligned streams, short last segment
        sym = (rs.rand(3, 2 * 32768 + 4099) < 0.45).astype(np.uint8)
        cum = [0, 2252, 4096]
    elif case == "segmented_q16":
        p = rs.dirichlet([0.5] * 16)
        sym = rs.choice(16, size=(2, 3 * 32768), p=p).astype(np.uint8)
        cum = range_coder.prob_to_cum_freq(p, resolution=1024)
    else:
        p = rs.dirichlet([0.3] * 256)
        sym = rs.choice(256, size=(2, 5003), p=p).astype(np.uint8)  # odd length: the unaligned symbol path
        cum = range_coder.prob_to_cum_freq(p * 0.999 + 0.001 / 256, resolution=65536)
    want = _host_streams(sym, cum)
    for src in (sym, torch.from_numpy(sym).cuda()):
        out, nbytes = codec.entropy_encode(src, cum)
        codec.check_status()
        out_h = out.cpu().numpy() if hasattr(out, "cpu") else out
        nb = nbytes.cpu().numpy() if hasattr(nbytes, "cpu") else nbytes
        for i in range(sym.shape[0]):
            assert bytes(out_h[i, :int(nb[i])]) == want[i], (case, i, int(nb[i]), len(want[i]))
        back = codec.entropy_decode(out, nbytes, sym.shape[1], cum)
        back = back.cpu().numpy() if hasattr(back, "cpu") else back
        assert np.array_equal(back, sym), case
    # and the host decoder reads the GPU's bytes
    dec = range_coder.decode_streams([bytes(out_h[i, :int(nb[i])]) for i in range(sym.shape[0])], [sym.shape[1]] * sym.shape[0], cum)
    assert all(np.array_equal(d, s) for d, s in zip(dec, sym))
    codec.close()


def test_entropy_stage_errors():
    codec, _, _ = make_codec("model_0", "fanin")
    sym = np.zeros((2, 64), np.uint8)
    sym[1, 5] = 3
    with pytest.raises(ValueError):
        codec.entropy_encode(sym, [0, 10, 16])           # symbol outside the table
    with pytest.raises(ValueError):
        codec.entropy_encode(sym[:1], [0, 0, 16])        # symbol of zero probability
    with pytest.raises(ValueError):
        codec.entropy_encode(sym[:1], [0, 10, 70000])    # total above 2^16
    with pytest.raises(ValueError):
        codec.entropy_encode(sym[:1], [1, 10, 16])
    out, nb = codec.entropy_encode(sym[:1], [0, 10, 16])
    assert int(nb[0]) <= out.shape[1]
    # corrupt streams (plain and segmented) stay in bounds and decode to what the host decoder makes of the same bytes
    rs = np.random.RandomState(8)
    for n in (4096, 2 * 32768 + 5):
        slot = int(codec.entropy_bound(n))
        buf = np.zeros((2, slot), np.uint8)
        nbytes = np.array([5000, 37], np.int64)
        for i in range(2):
            buf[i, :nbytes[i]] = rs.randint(0, 256, size=nbytes[i])
        got = codec.entropy_decode(buf, nbytes, n, [0, 2252, 4096])
        want = range_coder.decode_streams([bytes(buf[i, :nbytes[i]]) for i in range(2)], [n, n], [0, 2252, 4096])
        assert all(np.array_equal(g, w) for g, w in zip(got, want)), n
    codec.close()


def test_entropy_stage_full_size_and_entry_flows(tmp_path):
    """BASELINE config 2's symbol volume for 16 images (16 x 786 432 binary symbols): device-resident encode of the
    encoder's own output, byte identity with the host coder, decode back, timings printed; then entry.compress /
    uncompress with coder = gpu | host | serial write and read identical files."""
    codec, enc, dec = make_codec("model_0", "fanin", compute="tensor")
    rs = np.random.RandomState(11)
    imgs = torch.from_numpy(rs.randint(0, 256, size=(16, 1536, 2048, 3), dtype=np.uint8)).cuda()
    codec.hist_reset()
    sym = codec.encode_images(imgs, 128)                     # [16, 192, 8, 8, 64] in HBM
    counts = codec.hist_read()
    cum = entry.cum_freq_table(counts / counts.sum(), 4096)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out, nbytes = codec.entropy_encode(sym, cum)
    torch.cuda.synchronize()
    t_gpu = time.perf_counter() - t0
    codec.check_status()
    sym_h = sym.cpu().numpy().reshape(16, -1)
    t0 = time.perf_counter()
    want = _host_streams(sym_h, cum)
    t_host = time.perf_counter() - t0
    out_h, nb = out.cpu().numpy(), nbytes.cpu().numpy()
    for i in range(16):
        assert bytes(out_h[i, :int(nb[i])]) == want[i], i
    t0 = time.perf_counter()
    back = codec.entropy_decode(out, nbytes, sym_h.shape[1], cum)
    torch.cuda.synchronize()
    t_dec = time.perf_counter() - t0
    assert torch.equal(back.reshape(sym.shape), sym)
    print(f"[entropy stage] 16 streams x {sym_h.shape[1]} symbols: GPU encode {t_gpu * 1e3:.2f} ms, GPU decode {t_dec * 1e3:.2f} ms, "
          f"host thread pool encode {t_host * 1e3:.2f} ms; {int(nb.sum())} bytes ({8.0 * nb.sum() / (16 * 1536 * 2048):.4f} bpp)")
    # entry flows: three coders, identical files and reconstructions
    images = [O.synthetic_image(256, 384, 70 + i) for i in range(3)] + [O.synthetic_image(200, 300, 90)]
    names = [f"img_{i}" for i in range(4)]
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=128)
    prob = counts / counts.sum()
    outs = {c: entry.compress(codec, images, names, cfg, prob, str(tmp_path / c), coder=c) for c in ("gpu", "host", "serial")}
    for c in ("host", "serial"):
        for (p, n), (q, m) in zip(outs["gpu"], outs[c]):
            assert os.path.basename(p) == os.path.basename(q) and n == m and open(p, "rb").read() == open(q, "rb").read(), c
    recs = {c: entry.uncompress(codec, str(tmp_path / "gpu"), cfg, prob, coder=c) for c in ("gpu", "host", "serial")}
    for c in ("host", "serial"):
        assert all(np.array_equal(recs["gpu"][k], recs[c][k]) for k in recs["gpu"])
    assert sorted(recs["gpu"]) == names
    codec.close()


# ---- C-ABI plumbing (ADVICE r1) -----------------------------------------------------------------------------------
def test_stream_switch_orders_the_shared_workspaces():
    """tic_set_stream: work queued on the previous caller stream finishes before work on the next one touches the
    handle's workspaces (event ordering, no host sync): alternating streams gives the single-stream results."""
    codec, enc, dec = make_codec("model_0", "fanin", compute="tensor")
    rs = np.random.RandomState(5)
    imgs = torch.from_numpy(rs.randint(0, 256, size=(8, 512, 768, 3), dtype=np.uint8)).cuda()
    base = codec.encode_images(imgs, 128).clone()
    rec0 = codec.decode_images(base, 512, 768, 128).clone()
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    for it in range(6):
        with torch.cuda.stream(s1 if it % 2 == 0 else s2):
            sym = codec.encode_images(imgs, 128)
            outs.append((sym, codec.decode_images(sym, 512, 768, 128)))
    torch.cuda.synchronize()
    for sym, rec in outs:
        assert torch.equal(sym, base) and torch.equal(rec, rec0)
    codec.close()


def test_two_devices_in_one_process():
    """One handle per device, several devices per process: the per-device kernel attributes (dynamic shared memory
    limits) are configured on each device (ADVICE r1: a process-wide 'configured' flag skipped the second device)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gpurun --gpus 2)")
    enc, dec = params_for("model_0", "fanin")
    patches = patches_from_images(1, 256, 384, 128, seed=4)
    res = []
    for dev in (0, 1):
        for mode in ("fp32", "tensor"):
            c = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, enc_params=enc, dec_params=dec, compute=mode, device=dev)
            s = c.encode_patches(patches)
            res.append((s, c.decode_patches(s)))
            c.close()
    for s, r in res[1:]:
        assert (s != res[0][0]).mean() <= 1e-5 and float(np.abs(r - res[0][1]).max()) <= 1e-3
    assert np.array_equal(res[1][0], res[3][0]) and np.array_equal(res[1][1], res[3][1])  # tensor mode: device 0 == device 1


def test_shape_validation_raises_before_the_c_side_reads():
    codec, _, _ = make_codec("model_0", "fanin")
    with pytest.raises(ValueError):  # symbols of another variant (32 channels) for this codec
        codec.decode_images(np.zeros((1, 6, 8, 8, 32), np.uint8), 256, 384, 128)
    with pytest.raises(ValueError):  # wrong patch grid
        codec.decode_images(np.zeros((1, 5, 8, 8, 64), np.uint8), 256, 384, 128)
    with pytest.raises(ValueError):  # caller-supplied output of the wrong size
        codec.encode_images(np.zeros((1, 256, 384, 3), np.uint8), 128, out=np.zeros((1, 6, 8, 8, 32), np.uint8))
    with pytest.raises(ValueError):
        codec.roundtrip_images(np.zeros((1, 256, 384, 3), np.uint8), 128, out=np.zeros((1, 256, 380, 3), np.uint8))
    with pytest.raises(ValueError):
        codec.decode_patches(np.zeros((2, 8, 8, 64), np.uint8), out=np.zeros((2, 64, 64, 3), np.float32))
    codec.close()


# ---- the reference's unmodified entry points over the real Codec ---------------------------------------------------
def test_reference_entry_points_run_unmodified_on_the_gpu_codec(tmp_path):
    """encode.py:compress and decode.py:uncompress imported UNMODIFIED from a reference checkout (TIC_REFERENCE_ROOT, where
    one exists; tests/test_dropin.py runs the same scripts over the oracle adapter without a GPU) with
    tf_image_compression_b200.compat standing in for tensorflow / range_coder / skimage.io: files byte-identical to
    entry.compress, reconstructions identical to entry.uncompress, all three coders.  With or without a checkout, the
    entry flows over the GPU codec against the stored round trip (tests/golden/dropin_model0.npz)."""
    import test_dropin as D
    enc, dec, images, names, prob = D.dropin_case()
    codec = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, compute="tensor", seed=7)  # other weights: restored from the bundle
    if D.HAVE_REF:
        cfg, files, recs = D.run_reference_roundtrip(codec, tmp_path / "ref", images, names, prob, {**enc, **dec})
        D.check_against_entry_flows(codec, cfg, files, recs, images, names, prob, tmp_path, coders=("gpu", "host", "serial"))
    else:
        D.restore_from_checkpoint(codec, tmp_path / "ckpt", {**enc, **dec})
    D.check_against_stored(codec, images, names, prob, tmp_path / "golden", coders=("gpu", "host", "serial"))
    codec.close()
