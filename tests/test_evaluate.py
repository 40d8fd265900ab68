"""entry.evaluate on CPU with a stand-in codec: grouping by shape, input order, the set-level formulas of
processing_utils/evaluate.py, and the all-reduce of the integer sums over a world-size-2 gloo group."""
import os
import socket

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

from tf_image_compression_b200 import entry, parallel

CFG = {"patch_size": 128, "resolution": 4096}
PROB = [0.7, 0.3]


class StandInCodec:
    """Returns known integers instead of running the codec: the code size is a function of each image's first pixel,
    the squared error the exact one against a fixed 'reconstruction' (every pixel with its lowest bit flipped on
    the pixels whose value is a multiple of 3)."""

    def __init__(self):
        self.calls = []

    @staticmethod
    def recon(im):
        return np.where(im % 3 == 0, im ^ 1, im).astype(np.uint8)

    def evaluate_images(self, images, patch_size, cum_freq, out=None):
        self.calls.append((images.shape, int(patch_size), list(cum_freq)))
        code_bytes = np.array([100 + 7 * int(im[0, 0, 0]) + im.shape[1] for im in images], np.int64)
        sq_err = np.array([int(((im.astype(np.int64) - self.recon(im)) ** 2).sum()) for im in images], np.uint64)
        return code_bytes, sq_err, out


def _images():
    rs = np.random.RandomState(3)
    shapes = [(40, 60), (33, 17), (40, 60), (8, 8), (33, 17), (40, 60), (9, 12)]
    return [rs.randint(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in shapes]


def test_grouping_order_and_set_level_formulas():
    images = _images()
    codec = StandInCodec()
    res = entry.evaluate(codec, images, CFG, PROB)
    # one call per distinct shape, in order of first appearance, with the table of encode.py:76-91
    assert [c[0] for c in codec.calls] == [(3, 40, 60, 3), (2, 33, 17, 3), (1, 8, 8, 3), (1, 9, 12, 3)]
    cum = entry.cum_freq_table(PROB, 4096)
    assert all(c[1] == 128 and c[2] == cum for c in codec.calls)
    # per-image results in input order
    want_bytes = [100 + 7 * int(im[0, 0, 0]) + im.shape[1] for im in images]
    recons = [StandInCodec.recon(im) for im in images]
    want_se = [int(((im.astype(np.int64) - r) ** 2).sum()) for im, r in zip(images, recons)]
    assert res["code_bytes"].dtype == np.int64 and res["code_bytes"].tolist() == want_bytes
    assert res["sq_err"].dtype == np.uint64 and res["sq_err"].tolist() == want_se
    # evaluate.py's figures over the set, bit for bit what the host formulas give on files and reconstructions
    assert res["bpp"] == entry.bpp(want_bytes, images)
    assert res["psnr"] == entry.psnr(images, recons)
    hw = sum(im.shape[0] * im.shape[1] for im in images)
    assert res["bpp"] == 8.0 * sum(want_bytes) / hw
    assert res["psnr"] == 20.0 * np.log10(255.0) - 10.0 * np.log10(sum(want_se) / (3.0 * hw))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        images = _images()
        b, e = parallel.shard_range(len(images))
        res = entry.evaluate(StandInCodec(), images[b:e], CFG, PROB, group=dist.group.WORLD)
        local = entry.evaluate(StandInCodec(), images[b:e], CFG, PROB)
        q.put((rank, res["bpp"], res["psnr"], local["bpp"], local["psnr"], res["code_bytes"].tolist()))
    finally:
        dist.destroy_process_group()


def test_group_reduction_gives_dataset_wide_figures():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    whole = entry.evaluate(StandInCodec(), _images(), CFG, PROB)
    for _, bpp, psnr, local_bpp, local_psnr, _ in res:
        assert bpp == whole["bpp"] and psnr == whole["psnr"]      # every rank: the union's figures
        assert (local_bpp, local_psnr) != (whole["bpp"], whole["psnr"])  # not what one shard gives alone
    # per-image results stay per rank: the shards' concatenation is the whole list
    assert res[0][5] + res[1][5] == whole["code_bytes"].tolist()
