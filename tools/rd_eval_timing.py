"""Rate-distortion evaluation at BASELINE config 2 (model_0, 64 synthetic 2048x1536 images, P = 128, compute "tensor",
table from the encoder's own histogram):

  (a) Codec.evaluate_images, pinned host images, out=None: 604 MB H2D, 16 bytes per image D2H;
  (b) the same on device-resident images: nothing crosses PCIe but the 12-byte table and the results;
  (c) Codec.roundtrip_images alone on pinned host buffers (604 MB H2D + 604 MB D2H): the PCIe reference point;
  (d) encode + decode on device-resident images (roundtrip_images), the compute (b) adds the range coder and the
      squared error to.

Host clock around calls that end in a device synchronise; warm-up, then --reps repetitions, min / median / max.
Prints the card name and power limit, then checks entry.evaluate's bpp and PSNR against entry.bpp / entry.psnr
computed the slow way (files written by entry.compress, read back by entry.uncompress) on 4 of the images.
Writes nothing in the tree (the files go to a temporary directory).  Needs a B200; there is no fallback."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import tf_image_compression_b200 as T  # noqa: E402
from tf_image_compression_b200 import entry  # noqa: E402

MEAN = np.array([118.3, 113.9, 102.6], np.float32)
STD = np.array([61.7, 59.2, 63.8], np.float32)
H, W, P = 1536, 2048, 128


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the timing still stands; the card line says why it is missing
        return f"(nvidia-smi unavailable: {e})"


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts


def row(name, ts, h2d, d2h):
    ts = sorted(ts)
    print(f"{name:<44s} min {ts[0]:8.2f}  median {ts[len(ts) // 2]:8.2f}  max {ts[-1]:8.2f} ms   "
          f"H2D {h2d / 1e6:9.3f} MB  D2H {d2h / 1e6:9.3f} MB per step")
    return {"min_ms": ts[0], "median_ms": ts[len(ts) // 2], "max_ms": ts[-1]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    n = args.images
    dev = torch.device("cuda", 0)
    print(f"card: {card()}")
    g = torch.Generator().manual_seed(1234)
    host_img = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, generator=g).pin_memory()
    dev_img = host_img.to(dev)
    host_rec = torch.empty_like(host_img).pin_memory()
    codec = T.Codec("model_0", quan_scale=2, mean=MEAN, std=STD, compute="tensor", seed=1234)
    codec.hist_reset()
    codec.encode_images(dev_img, P)
    counts = codec.hist_read().astype(np.float64)
    prob = counts / counts.sum()
    cfg = dict(entry.DEFAULT_CONFIG, patch_size=P)
    cum = entry.cum_freq_table(prob, int(cfg["resolution"]))
    img_bytes = n * H * W * 3
    table_bytes = 4 * len(cum)
    print(f"workload: model_0, {n} x {W}x{H} uniform-random images, P = {P}, compute tensor; table {list(cum)}")

    res = {}
    res["a"] = row("(a) evaluate_images, pinned host", timed(lambda: codec.evaluate_images(host_img, P, cum), args.warmup, args.reps),
                   img_bytes + table_bytes, 16 * n)
    res["b"] = row("(b) evaluate_images, device-resident", timed(lambda: codec.evaluate_images(dev_img, P, cum), args.warmup, args.reps),
                   table_bytes, 0)
    res["b_kernel_ms"] = codec.last_kernel_ms()
    res["c"] = row("(c) roundtrip_images, pinned host", timed(lambda: codec.roundtrip_images(host_img, P, out=host_rec, want_symbols=False),
                                                              args.warmup, args.reps), img_bytes, img_bytes)
    res["d"] = row("(d) roundtrip_images, device-resident", timed(lambda: codec.roundtrip_images(dev_img, P), args.warmup, args.reps), 0, 0)
    print(f"(b) device time of the last call's kernel sequence (tic_last_kernel_ms): {res['b_kernel_ms']:.2f} ms")
    codec.check_status()

    cb, se, _ = codec.evaluate_images(host_img, P, cum)
    hw = n * H * W
    print(f"batch: {int(cb.sum())} bytes, bpp {8.0 * cb.sum() / hw:.6f}, "
          f"PSNR {20 * np.log10(255.0) - 10 * np.log10(float(se.sum()) / (3 * hw)):.6f} dB")

    # the slow way on 4 images: files, reconstructions, host formulas
    imgs = [host_img[i].numpy() for i in range(min(4, n))]
    names = [f"img_{i}" for i in range(len(imgs))]
    with tempfile.TemporaryDirectory() as tmp:
        files = entry.compress(codec, imgs, names, cfg, prob, tmp, coder="host")
        recs = entry.uncompress(codec, tmp, cfg, prob)
    slow_bpp = entry.bpp([nb for _, nb in files], imgs)
    slow_psnr = entry.psnr(imgs, [recs[k] for k in names])
    fast = entry.evaluate(codec, imgs, cfg, prob)
    ok = fast["bpp"] == slow_bpp and fast["psnr"] == slow_psnr
    print(f"4 images: entry.evaluate bpp {fast['bpp']!r} PSNR {fast['psnr']!r}; files + host formulas bpp {slow_bpp!r} "
          f"PSNR {slow_psnr!r}: {'identical' if ok else 'DIFFERENT'}")
    codec.close()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
