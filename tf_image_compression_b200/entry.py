"""The reference's entry-point flows on top of the B200 path: compress (encode.py:125-212), uncompress
(decode.py:143-251, with the submit/2 post-filter call order submit/2/decoder.py:183-198), the one-graph round
trip (test.py:95-146) and the dataset-wide
symbol table (get_encoded_distribution.py:85-155).  File names, config keys, table construction and the
bitstream order (patch-major, then h, w, c: encode.py:171-182) are the reference's; images are processed in
batches through Codec.encode_images / decode_images instead of one sess.run per 64 patches."""
from __future__ import annotations

import os
from pathlib import Path

import numpy as np

from . import parallel, range_coder

DEFAULT_CONFIG = {"name_sep": "@_@", "resolution": 4096, "patch_size": 128, "quan_scale": 2}  # model_N/config.json keys


def cum_freq_table(prob, resolution):
    """encode.py:76-91 == decode.py:79-93: freq = prob * resolution + 1 (no zero-probability symbol), renormalise,
    range_coder.prob_to_cum_freq(modified_prob, resolution)."""
    prob = np.asarray(prob, dtype=np.float64)
    modified_freq = prob * resolution + 1
    modified_prob = modified_freq / np.sum(modified_freq)
    return range_coder.prob_to_cum_freq(modified_prob, resolution=resolution)


def encoded_name(image_name, image_shape, seq_data_len, encoded_patches_shape, config):
    """encode.py:102-122: '<name>@_@<eh>_<ew>_<ec>@_@<len>_<H>_<W>.encoded'."""
    sep = config["name_sep"]
    stem = str(image_name).split("/")[-1].replace(".png", "")
    eh, ew, ec = encoded_patches_shape
    height, width = image_shape[0], image_shape[1]
    return f"{stem}{sep}{eh}_{ew}_{ec}{sep}{seq_data_len}_{height}_{width}.encoded"


def parse_encoded_name(filename, config):
    """decode.py:104-140: -> (stem, (eh, ew, ec), seq_data_len, height, width)."""
    sep = config["name_sep"]
    parts = str(filename).replace(".encoded", "").split(sep)
    if len(parts) < 3:
        raise ValueError(f"not an encoded file name: {filename!r}")
    eh, ew, ec = (int(v) for v in parts[1].split("_"))
    n, h, w = (int(v) for v in parts[-1].split("_"))
    return parts[0], (eh, ew, ec), n, h, w


def compress(codec, images, names, config, prob, output_dir, coder="host"):
    """Encode a list of uint8 [H,W,3] images (any sizes) and write one range-coded file per image.
    Images of equal size go through the codec as one batch; their per-image streams are coded concurrently —
    coder="host": range_coder.encode_streams (thread pool), coder="gpu": Codec.entropy_encode (symbols never leave the
    device, only the compressed bytes come back), coder="serial": one RangeEncoder per file like encode.py:186-202.
    The three write identical files.  Returns [(path, n_bytes)] in input order."""
    P = int(config["patch_size"])
    cum = cum_freq_table(prob, int(config["resolution"]))
    out = [None] * len(images)
    os.makedirs(output_dir, exist_ok=True)
    by_shape = {}
    for i, im in enumerate(images):
        by_shape.setdefault(tuple(im.shape), []).append(i)
    hb, wb, cb = codec.bottleneck_shape(P)
    for shape, idx in by_shape.items():
        batch = np.ascontiguousarray(np.stack([images[i] for i in idx]), dtype=np.uint8)
        if coder == "gpu":
            import torch
            dev = torch.device("cuda", codec.device)
            sym = codec.encode_images(torch.from_numpy(batch).to(dev), P)  # stays in HBM
            packed, nbytes = codec.entropy_encode(sym, cum)
            nbytes = nbytes.cpu().numpy()
            codec.check_status()
            packed = packed.cpu().numpy()
            blobs = [packed[k, :int(nbytes[k])].tobytes() for k in range(len(idx))]
            seq_len = int(np.prod(sym.shape[1:]))
        else:
            sym = codec.encode_images(batch, P)  # [B, gh*gw, hb, wb, cb] uint8, patch-major
            seq_len = int(np.prod(sym.shape[1:]))
            blobs = range_coder.encode_streams(sym.reshape(len(idx), -1), cum) if coder == "host" else None
        for k, i in enumerate(idx):
            path = str(Path(output_dir) / encoded_name(names[i], shape, seq_len, (hb, wb, cb), config))
            if blobs is None:
                enc = range_coder.RangeEncoder(path)
                enc.encode(sym[k].reshape(-1), cum)
                enc.close()
                out[i] = (path, enc.bytes_written)
            else:
                with open(path, "wb") as f:
                    f.write(blobs[k])
                out[i] = (path, len(blobs[k]))
    return out


def uncompress(codec, input_dir, config, prob, postfilter=False, coder="host"):
    """Decode every '*.encoded' file of input_dir -> {stem: uint8 [H,W,3]} (np.around of the stitched float image,
    decode.py:249; with postfilter=True the float image goes through rmbe first, submit/2/decoder.py:183-198).
    coder="host": all files of a shape group decoded concurrently (range_coder.decode_streams); "gpu": Codec.entropy_decode
    (the compressed bytes go up, symbols are produced in HBM); "serial": one RangeDecoder per file like decode.py:182."""
    P = int(config["patch_size"])
    cum = cum_freq_table(prob, int(config["resolution"]))
    files = sorted(f for f in os.listdir(input_dir) if f.endswith(".encoded"))
    groups = {}
    want = tuple(codec.bottleneck_shape(P))
    for f in files:
        stem, eshape, n, h, w = parse_encoded_name(f, config)
        if tuple(eshape) != want:
            raise ValueError(f"{f}: encoded patch shape {tuple(eshape)} is not this codec's {want} at patch size {P} "
                             "(file of another model variant / patch size?)")
        if n != (-(-h // P)) * (-(-w // P)) * eshape[0] * eshape[1] * eshape[2]:
            raise ValueError(f"{f}: sequence length {n} does not match a {h}x{w} image in {P}x{P} patches")
        if coder == "serial":
            dec = range_coder.RangeDecoder(str(Path(input_dir) / f))
            seq = dec.decode(n, cum, dtype=np.uint8)
            dec.close()
        else:
            with open(Path(input_dir) / f, "rb") as fh:
                seq = fh.read()  # the stored bytes; decoded per shape group below
        groups.setdefault((h, w, eshape), []).append((stem, seq))
    result = {}
    for (h, w, eshape), items in groups.items():
        gh, gw = -(-h // P), -(-w // P)
        n = gh * gw * eshape[0] * eshape[1] * eshape[2]
        if coder == "host":
            seqs = range_coder.decode_streams([b for _, b in items], [n] * len(items), cum)
            items = [(stem, s) for (stem, _), s in zip(items, seqs)]
        elif coder == "gpu":
            import torch
            stride = max(16, -(-max(len(b) for _, b in items) // 16) * 16)
            packed = np.zeros((len(items), stride), np.uint8)
            for k, (_, b) in enumerate(items):
                packed[k, :len(b)] = np.frombuffer(b, np.uint8)
            dev = torch.device("cuda", codec.device)
            d_sym = codec.entropy_decode(torch.from_numpy(packed).to(dev), torch.tensor([len(b) for _, b in items]), n, cum)
            seqs = d_sym.cpu().numpy()
            items = [(stem, seqs[k]) for k, (stem, _) in enumerate(items)]
        sym = np.stack([s.reshape(gh * gw, *eshape) for _, s in items])
        if postfilter:
            rec = codec.decode_images(sym, h, w, P, out_dtype=np.float32)
            codec.postfilter_images(rec)
            rec = codec.round_u8(rec)
        else:
            rec = codec.decode_images(sym, h, w, P, out_dtype=np.uint8)
        for k, (stem, _) in enumerate(items):
            result[stem] = rec[k]
    return result


def compress_and_uncompress(codec, images, config):
    """test.py:95-146: encoder and decoder in one graph, no bitstream — the reference's quality check.  Images of
    equal size go through Codec.roundtrip_images as one batch.  Returns the uint8 reconstructions in input order
    (io.imsave of the stitched float image rounds like decode.py:249)."""
    P = int(config["patch_size"])
    out = [None] * len(images)
    by_shape = {}
    for i, im in enumerate(images):
        by_shape.setdefault(tuple(im.shape), []).append(i)
    for shape, idx in by_shape.items():
        batch = np.ascontiguousarray(np.stack([images[i] for i in idx]), dtype=np.uint8)
        rec, _ = codec.roundtrip_images(batch, P, want_symbols=False)
        for k, i in enumerate(idx):
            out[i] = rec[k]
    return out


def get_distribution(codec, patches, group=None):
    """get_encoded_distribution.py:85-155 over this rank's shard of the patch list: encode (the histogram is fused
    into the bottleneck epilogue), all-reduce the q counts over the ranks, prob = freq / sum(freq)."""
    codec.hist_reset()
    if len(patches):
        codec.encode_patches(patches)
    return parallel.distribution(parallel.allreduce_histogram(codec, group))


def cal_distribution(codec, patches, batch_size=64):
    """cal_encoded_distribution.py:78-160 over a patch list: the float64 running mean of every bottleneck position,
    folded in one sess.run batch of 64 at a time exactly as the reference does it (:111-128: seq_prob = seq_prob *
    (prev_n / n) + np.sum(batch, axis=0) / n, the batch sum and its division in float32 like the fetched tensor),
    prob = [1 - mean(seq_prob), mean(seq_prob)] (:144-145) and encoded_order = the stable sort of the positions by
    seq_prob (:149).  The device supplies exact integer per-batch sums (tic_position_sums_batched); the floating-point
    folding is the reference's own expression.  Returns (prob float64[2], encoded_order int list, seq_prob float64[npos])
    — what the script saves as distribution_info_N.npy / order_info_N.npy."""
    hb, wb, cb = codec.bottleneck_shape(int(patches.shape[1]))
    npos = hb * wb * cb
    seq_prob = np.zeros(npos)
    n = 0
    if len(patches):
        sym = codec.encode_patches(patches)
        sums = codec.position_sums_batched(sym, batch_size)
        sums = sums.cpu().numpy() if hasattr(sums, "cpu") else sums
        for b in range(sums.shape[0]):
            batch_num = min(batch_size, len(patches) - b * batch_size)
            prev_n = n
            n += batch_num
            batch_sum = sums[b].astype(np.float32)  # np.sum of the fetched float32 symbols: exact (<= 64 * (q - 1))
            seq_prob = seq_prob * (1.0 * prev_n / n) + batch_sum / n
    one_prob = np.mean(seq_prob)
    prob = [1.0 - one_prob, one_prob]
    encoded_order = sorted(range(len(seq_prob)), key=lambda k: seq_prob[k])
    return np.asarray(prob), encoded_order, seq_prob


def evaluate(codec, images, config, prob, group=None):
    """scipt_bash/encode_decode_evaluate.sh without files: encode.py + decode.py + processing_utils/evaluate.py over a list
    of uint8 [H,W,3] images (any sizes), on the device (Codec.evaluate_images per group of equal-sized images, the table
    of encode.py:76-91).  Returns {"bpp", "psnr", "code_bytes", "sq_err"}: the set-level figures of evaluate.py (:10-49)
    computed from exact integer sums in the float64 expressions of bpp() / psnr(), and the per-image file sizes and
    integer squared errors in input order.  With `group`, the sums are all-reduced over its ranks first, so every rank
    returns the figures of the whole dataset (the PSNR of a union is not a function of the per-rank PSNRs)."""
    P = int(config["patch_size"])
    cum = cum_freq_table(prob, int(config["resolution"]))
    code_bytes = np.zeros(len(images), np.int64)
    sq_err = np.zeros(len(images), np.uint64)
    by_shape = {}
    for i, im in enumerate(images):
        by_shape.setdefault(tuple(im.shape), []).append(i)
    for shape, idx in by_shape.items():
        batch = np.ascontiguousarray(np.stack([images[i] for i in idx]), dtype=np.uint8)
        nb, se, _ = codec.evaluate_images(batch, P, cum)
        code_bytes[idx] = nb
        sq_err[idx] = se
    pixels = sum(int(im.shape[0]) * int(im.shape[1]) for im in images)
    totals = np.array([int(code_bytes.sum()), int(sq_err.sum()), pixels, 3 * pixels], np.int64)
    if group is not None:
        totals = parallel.allreduce_counts(totals, group)
    n_bytes, se, hw, hwc = (int(v) for v in totals)
    return {"bpp": 8.0 * float(n_bytes) / float(hw),
            "psnr": 20.0 * np.log10(255.0) - 10.0 * np.log10(float(se) / hwc),
            "code_bytes": code_bytes, "sq_err": sq_err}


def psnr(originals, reconstructions):
    """processing_utils/evaluate.py:10-30: 20 log10(255) - 10 log10(sum SE / sum HWC) over the whole set."""
    se, cnt = 0.0, 0
    for a, b in zip(originals, reconstructions):
        d = a.astype(np.float64) - b.astype(np.float64)
        se += float((d * d).sum())
        cnt += d.size
    return 20.0 * np.log10(255.0) - 10.0 * np.log10(se / cnt)


def bpp(n_bytes_list, images):
    """processing_utils/evaluate.py:33-49: 8 * sum(file bytes) / sum(H * W)."""
    return 8.0 * float(sum(n_bytes_list)) / float(sum(im.shape[0] * im.shape[1] for im in images))
