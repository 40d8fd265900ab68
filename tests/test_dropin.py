"""The drop-in claim (north_star: "encode.py / decode.py ... stay unchanged"): the reference's UNMODIFIED entry points,
imported from the reference checkout named by TIC_REFERENCE_ROOT with `tensorflow`, `range_coder` and `skimage.io` stood in by
tf_image_compression_b200.compat, run compress() then uncompress() on synthetic images, and their files / reconstructions
are compared byte for byte with entry.compress / entry.uncompress over the same codec.

The reference is not part of this repository.  tests/golden/dropin_model0.npz stores the round trip of the same inputs
(file names, file bytes, symbols, reconstructions), so the comparison runs without a checkout too; with one, the
reference's output is checked against the entry flows and the stored round trip alike.

Here the codec is the oracle adapter (tests/oracle_codec.py): that pins the whole host side (compat, model_api, entry,
range_coder, checkpoint, file naming).  tests/test_gpu_parity2.py runs the same comparison over the real Codec, and the
GPU parity tests pin Codec == oracle."""
import argparse
import json
import os
from pathlib import Path

import numpy as np

from oracle import codec_oracle as O
from tf_image_compression_b200 import checkpoint as K
from tf_image_compression_b200 import compat, entry, range_coder

# a checkout of the reference project (bolin-chen/tf_image_compression); it is not part of this repository, so the
# reference's scripts run only where TIC_REFERENCE_ROOT names one
REF = Path(os.environ["TIC_REFERENCE_ROOT"]) if os.environ.get("TIC_REFERENCE_ROOT") else None
HAVE_REF = REF is not None and (REF / "encode.py").is_file()
GOLDEN = Path(__file__).parent / "golden" / "dropin_model0.npz"
MEAN = np.array([118.3, 113.9, 102.6], np.float32)
STD = np.array([61.7, 59.2, 63.8], np.float32)


def dropin_case():
    """The round trip's inputs: model_0 fan-in weights (seeds 1234 / 1235), two synthetic images (the second needs
    reflect padding at P = 256), their names and the two-symbol table."""
    ov = O.VARIANTS["model_0"]
    enc = O.init_params(ov["enc"], 3, 1234, "fanin")
    dec = O.condition_decoder("model_0", O.init_params(ov["dec"], ov["bottleneck"], 1235, "fanin"), 2)
    images = [O.synthetic_image(256, 512, 3), O.synthetic_image(300, 260, 4)]
    return enc, dec, images, ["kodim_a", "kodim_b"], np.array([0.55, 0.45])


def restore_from_checkpoint(codec, root, params, model_num=0):
    """What the reference's flow does before compress(): write model_N/params_for_test/params as a TF-V2 bundle under
    `root`, then utils.restore_params (checkpoint.restore_params) into the codec."""
    K.write_checkpoint(str(Path(root) / f"model_{model_num}" / "params_for_test" / "params"), params)
    K.restore_params(codec, model_num=model_num, root=str(root))


def stored_roundtrip():
    """tests/golden/dropin_model0.npz (tests/golden/make_golden.py) -> (config, [(file name, file bytes, symbols,
    reconstruction)] in image order)."""
    z = np.load(GOLDEN)
    cfg = json.loads(str(z["config_json"]))
    out = []
    for i, name in enumerate(z["file_names"]):
        name = str(name)
        n = entry.parse_encoded_name(name, cfg)[2]
        out.append((name, z[f"file_{i}"].tobytes(), np.unpackbits(z[f"symbols_{i}"], count=n), z[f"recon_{i}"]))
    return cfg, out


def check_against_stored(codec, images, names, prob, work, coders=("host", "serial")):
    """entry.compress / entry.uncompress over `codec` against the stored round trip.  The stored files are the stored
    symbols range-coded; the codec's files carry the stored names, hold the stored symbols up to one per image (a logit
    within rounding noise of the quantiser threshold may fall either way on other hardware) and equal the stored files
    byte for byte wherever the symbols are equal; every coder decodes the stored files to within one grey level of the
    stored reconstructions (rate < 1e-4).  Returns the stored config."""
    cfg, stored = stored_roundtrip()
    work = Path(work)
    cum = entry.cum_freq_table(prob, cfg["resolution"])
    for name, blob, sym, _ in stored:
        assert range_coder.encode_streams([sym], cum)[0] == blob, name
    out = entry.compress(codec, images, names, cfg, prob, str(work / "own"), coder=coders[0])
    assert [os.path.basename(p) for p, _ in out] == [s[0] for s in stored]
    for (p, nbytes), (name, blob, sym, _) in zip(out, stored):
        own = open(p, "rb").read()
        own_sym = range_coder.decode_streams([own], [sym.size], cum)[0]
        assert nbytes == len(own) and int((own_sym != sym).sum()) <= 1, name
        assert own == blob or not np.array_equal(own_sym, sym), name
    for c in coders[1:]:
        other = entry.compress(codec, images, names, cfg, prob, str(work / ("own_" + c)), coder=c)
        for (p, _), (q, _) in zip(out, other):
            assert open(p, "rb").read() == open(q, "rb").read(), c
    src = work / "stored"
    src.mkdir(parents=True)
    for name, blob, _, _ in stored:
        (src / name).write_bytes(blob)
    for c in coders:
        recs = entry.uncompress(codec, str(src), cfg, prob, coder=c)
        assert sorted(recs) == sorted(names)
        for nm, im, (_, _, _, want) in zip(names, images, stored):
            d = np.abs(recs[nm].astype(int) - want.astype(int))
            assert recs[nm].shape == im.shape and d.max() <= 1 and (d != 0).mean() < 1e-4, (c, nm)
    return cfg


def run_reference_roundtrip(codec, work, images, names, prob, ckpt_params, model_num=0):
    """Lay out a reference working directory (config.json copied verbatim, distribution table, image list, PNG
    inputs, model_N/params_for_test/params as a TF-V2 bundle), then call the unmodified compress() and uncompress()."""
    from PIL import Image
    work = Path(work)
    (work / f"model_{model_num}").mkdir(parents=True)
    (work / "data_info").mkdir()
    (work / "images").mkdir()
    cfg_text = (REF / f"model_{model_num}" / "config.json").read_text()
    (work / f"model_{model_num}" / "config.json").write_text(cfg_text)
    np.save(work / "data_info" / f"distribution_info_{model_num}.npy", prob)
    paths = []
    for im, nm in zip(images, names):
        p = work / "images" / (nm + ".png")
        Image.fromarray(im).save(p)
        paths.append(str(p))
    (work / "data_info" / "list.txt").write_text("\n".join(paths) + "\n")
    (work / f"model_{model_num}" / "params_for_test").mkdir()
    K.write_checkpoint(str(work / f"model_{model_num}" / "params_for_test" / "params"), ckpt_params)
    cwd = os.getcwd()
    os.chdir(work)
    try:
        with compat.installed(codec, reference_root=str(REF)):
            enc = compat.load_entry(REF / "encode.py")
            dec = compat.load_entry(REF / "decode.py")
            args = argparse.Namespace(model_num=str(model_num), gpu_num="0", debug_mode="off", params_file="",
                                      data_list="data_info/list.txt", output_dir="model_{}/encoded_data")
            enc.compress(compat.Session(), compat.model_module(model_num), args)
            dargs = argparse.Namespace(model_num=str(model_num), gpu_num="0", debug_mode="off", params_file="",
                                       input_dir="model_{}/encoded_data", output_dir="model_{}/recons_data")
            dec.uncompress(compat.Session(), compat.model_module(model_num), dargs)
    finally:
        os.chdir(cwd)
    enc_dir = work / f"model_{model_num}" / "encoded_data"
    rec_dir = work / f"model_{model_num}" / "recons_data"
    files = {f: (enc_dir / f).read_bytes() for f in sorted(os.listdir(enc_dir))}
    recs = {f[:-4]: np.asarray(Image.open(rec_dir / f)) for f in sorted(os.listdir(rec_dir))}
    return json.loads(cfg_text), files, recs


def check_against_entry_flows(codec, cfg, files, recs, images, names, prob, tmp_path, coders=("host", "serial")):
    """entry.compress / entry.uncompress over the same codec: byte-identical files, identical reconstructions."""
    out = entry.compress(codec, images, names, cfg, prob, str(tmp_path / "own"), coder=coders[0])
    assert sorted(os.path.basename(p) for p, _ in out) == sorted(files)
    for p, nbytes in out:
        assert open(p, "rb").read() == files[os.path.basename(p)] and nbytes == len(files[os.path.basename(p)])
    for c in coders[1:]:
        other = entry.compress(codec, images, names, cfg, prob, str(tmp_path / ("own_" + c)), coder=c)
        for (p, _), (q, _) in zip(out, other):
            assert open(p, "rb").read() == open(q, "rb").read(), c
    for c in coders:
        own = entry.uncompress(codec, str(tmp_path / "own"), cfg, prob, coder=c)
        assert sorted(own) == sorted(recs) == sorted(names)
        for nm, im in zip(names, images):
            assert recs[nm].shape == im.shape and np.array_equal(own[nm], recs[nm]), (c, nm)
    # file names carry the reference's metadata (encode.py:102-122)
    P = cfg["patch_size"]
    for f in files:
        stem, eshape, n, h, w = entry.parse_encoded_name(f, cfg)
        assert n == (-(-h // P)) * (-(-w // P)) * eshape[0] * eshape[1] * eshape[2]


def test_reference_entry_points_run_unmodified_on_the_oracle_codec(tmp_path):
    """With a reference checkout: its compress() / uncompress() over the oracle codec == entry.compress / uncompress.
    With or without one: the entry flows against the stored round trip of the same inputs."""
    from oracle_codec import OracleCodec
    ov = O.VARIANTS["model_0"]
    enc, dec, images, names, prob = dropin_case()
    # the codec starts from OTHER weights: the flow itself must restore the checkpoint (utils.restore_params)
    codec = OracleCodec("model_0", 2, MEAN, STD, O.init_params(ov["enc"], 3, 99, "fanin"),
                        O.init_params(ov["dec"], ov["bottleneck"], 98, "fanin"))
    if HAVE_REF:
        cfg, files, recs = run_reference_roundtrip(codec, tmp_path / "ref", images, names, prob, {**enc, **dec})
        assert cfg["patch_size"] == 256 and cfg["quan_scale"] == 2  # the reference's own model_0/config.json
        # one sess.run per <= 64 patches, like the reference (2 and 4 patches here)
        assert ("encode_patches", 2) in codec.calls and ("encode_patches", 4) in codec.calls
        assert ("decode_patches", 2) in codec.calls and ("decode_patches", 4) in codec.calls
        check_against_entry_flows(codec, cfg, files, recs, images, names, prob, tmp_path)
    else:
        restore_from_checkpoint(codec, tmp_path / "ckpt", {**enc, **dec})
    assert all(np.array_equal(codec.enc_params[k], enc[k]) for k in enc)  # restore_params replaced the weights
    assert all(np.array_equal(codec.dec_params[k], dec[k]) for k in dec)
    stored_cfg = check_against_stored(codec, images, names, prob, tmp_path / "golden")
    if HAVE_REF:  # the stored config is the reference's, as far as the flows read it
        assert {k: cfg[k] for k in stored_cfg} == stored_cfg
    assert all(entry.parse_encoded_name(s[0], stored_cfg)[1] == (16, 16, 64) for s in stored_roundtrip()[1])


def test_uncompress_with_postfilter_on_the_oracle_codec(tmp_path):
    """The submit/2 decode flow (decode -> stitch -> rmbe -> np.around, submit/2/decoder.py:183-198) through
    entry.uncompress(postfilter=True) over the oracle codec of model_3, with the host and the serial coder: it equals
    the oracle chain composed by hand from the symbols, exactly; postfilter=False equals decode_images(..., uint8).
    200x300 is a multiple neither of the 128-pixel patch nor of the rmbe tile grid."""
    from oracle_codec import OracleCodec
    from gpu_common import PM, PS, post_params
    ov = O.VARIANTS["model_3"]
    enc = O.init_params(ov["enc"], 3, 1234, "fanin")
    dec = O.condition_decoder("model_3", O.init_params(ov["dec"], ov["bottleneck"], 1235, "fanin"), 2)
    pp = post_params()
    codec = OracleCodec("model_3", 2, MEAN, STD, enc, dec, post_params=pp, post_mean=PM, post_std=PS)
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=128)
    P, prob = cfg["patch_size"], np.array([0.55, 0.45])
    images = {"a": O.synthetic_image(256, 384, 11), "b": O.synthetic_image(200, 300, 12)}
    entry.compress(codec, list(images.values()), list(images), cfg, prob, str(tmp_path), coder="host")
    want, plain = {}, {}
    for nm, im in images.items():
        H, W, _ = im.shape
        sym = codec.encode_images(im[None], P)[0]
        stitched = O.concat_patches(list(O.decoder(sym, "model_3", dec, MEAN, STD, 2)), H, W, P)
        want[nm] = O.around_u8(O.rmbe(stitched, lambda t: O.postfilter(t, "rmbe", pp, PM, PS)))
        plain[nm] = codec.decode_images(sym[None], H, W, P)[0]
        assert not np.array_equal(want[nm], plain[nm])  # the filter changes the image
    for c in ("host", "serial"):
        got = entry.uncompress(codec, str(tmp_path), cfg, prob, postfilter=True, coder=c)
        got_plain = entry.uncompress(codec, str(tmp_path), cfg, prob, coder=c)
        for nm in images:
            assert got[nm].dtype == np.uint8 and np.array_equal(got[nm], want[nm]), (c, nm)
            assert np.array_equal(got_plain[nm], plain[nm]), (c, nm)
