"""Host-side handle over the C ABI: one Codec per GPU, mirroring what the reference builds per
process (graph + restored params + one tf.Session, encode.py:125-149 / decode.py:143-169)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from . import variants as V

try:  # torch is plumbing only (device buffers, streams, distributed)
    import torch
except Exception:  # pragma: no cover
    torch = None


class TicError(RuntimeError):
    pass


def inverse_sigmoid_lut(quan_scale: int) -> np.ndarray:
    """q-entry table of the decoder's first op, evaluated in fp32 in the reference's op order:
    basic_block.reverse_sigmoid((input + 1e-6) / (quan_scale - 1 + 1e-5))  (model_0/model.py:153,
    basic_block/basic_block.py:152-155)."""
    s = np.arange(quan_scale, dtype=np.float32)
    p = (s + np.float32(1e-6)) / np.float32(quan_scale - 1 + 1e-5)
    return np.log(p / (np.float32(1.0) - p)).astype(np.float32)


def reference_init(layers, seed=1234):
    """Random stand-in for an absent checkpoint, following the reference initialisers:
    tf.random_normal_initializer(0, 0.01) kernels, zero biases (model_0/model.py:57-58)."""
    rs = np.random.RandomState(seed)
    params = {}
    for l in layers:
        params[l.scope + "/kernel"] = rs.normal(0.0, 0.01, size=l.kernel_shape).astype(np.float32)
        params[l.scope + "/bias"] = np.zeros(l.cout, dtype=np.float32)
    return params


def _is_torch(x):
    return torch is not None and isinstance(x, torch.Tensor)


class _Buf:
    """Pointer + placement of a numpy array or a torch tensor (CPU or CUDA), kept alive while in use."""

    def __init__(self, x, dtype, device_index, codec=None):
        if codec is not None and _is_torch(x) and x.is_cuda:
            codec._follow_torch_stream()
        self.keep = x
        if _is_torch(x):
            want = {np.uint8: torch.uint8, np.float32: torch.float32}[dtype]
            if x.dtype != want:
                raise ValueError(f"expected {want}, got {x.dtype}")
            if not x.is_contiguous():
                raise ValueError("tensor must be contiguous")
            if x.is_cuda:
                if x.device.index != device_index:
                    raise ValueError(f"tensor is on {x.device}, codec is on cuda:{device_index}")
                self.mem = L.MEM_DEVICE
            else:
                self.mem = L.MEM_HOST
            self.ptr = x.data_ptr()
        else:
            a = x
            if a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
                raise ValueError(f"expected C-contiguous {np.dtype(dtype)}, got {a.dtype}")
            self.mem = L.MEM_HOST
            self.ptr = a.ctypes.data


class Codec:
    """B200 codec handle for one model variant.

    variant: a key of variants.VARIANTS ('model_0', 'base_model/ch_128', …)
    quan_scale: config.json 'quan_scale'
    mean/std: channel_normalization_params.npz (0..255 scale, shape [3])
    enc_params/dec_params: {'<scope>/kernel', '<scope>/bias'} fp32 arrays in the TF variable layouts;
        None -> reference initialisers (seeded)."""

    def __init__(self, variant, quan_scale=2, mean=(0.0, 0.0, 0.0), std=(1.0, 1.0, 1.0), enc_params=None,
                 dec_params=None, bottleneck_channel=None, device=0, compute="fp32", seed=1234):
        self._h = None
        self.lib = L.load()
        custom = variant if isinstance(variant, dict) else None  # {'encoder': table, 'decoder': table, 'bottleneck_channel': c}
        self.variant = "custom" if custom else V.resolve(variant)
        self.quan_scale = int(quan_scale)
        self.device = int(device)
        h = C.c_void_p()
        rc = self.lib.tic_create(C.byref(h), self.device)
        if rc != L.OK:
            raise TicError(f"tic_create failed ({rc}): {self.lib.tic_create_error().decode()}")
        self._h = h
        if custom:
            cb = bottleneck_channel or custom["bottleneck_channel"]
            self.enc_layers = V.primitive_layers(custom["encoder"], 3, cb)
            self.dec_layers = V.primitive_layers(custom["decoder"], cb, cb)
        else:
            self.enc_layers = V.encoder_layers(self.variant, bottleneck_channel)
            self.dec_layers = V.decoder_layers(self.variant, bottleneck_channel)
        self.post_layers = None
        self.mean = np.asarray(mean, dtype=np.float32).reshape(3)
        self.std = np.asarray(std, dtype=np.float32).reshape(3)
        self._set_graph(L.GRAPH_ENCODER, self.enc_layers, enc_params if enc_params is not None
                        else reference_init(self.enc_layers, seed))
        self._set_graph(L.GRAPH_DECODER, self.dec_layers, dec_params if dec_params is not None
                        else reference_init(self.dec_layers, seed + 1))
        for g in (L.GRAPH_ENCODER, L.GRAPH_DECODER):
            self._check(self.lib.tic_set_norm(self._h, g, self.mean.ctypes.data, self.std.ctypes.data))
        lut = inverse_sigmoid_lut(self.quan_scale)
        self._check(self.lib.tic_set_quantizer(self._h, self.quan_scale, lut.ctypes.data))
        self.set_compute(compute)

    # ---- plumbing ------------------------------------------------------------------------------
    def _check(self, rc):
        if rc == L.OK:
            return
        msg = self.lib.tic_last_error(self._h).decode()
        if rc == L.ERR_INVALID:
            raise ValueError(msg)
        raise TicError(f"tic error {rc}: {msg}")

    def _set_graph(self, gid, layers, params):
        arr = (L.LayerDesc * len(layers))()
        for i, l in enumerate(layers):
            arr[i] = L.LayerDesc(L.CONV if l.kind == "c" else L.DECONV, l.cin, l.cout, l.stride,
                                 L.ACT_RELU if l.act == V.RELU else L.ACT_IDENTITY, l.res_begin, l.res_end)
        self._check(self.lib.tic_set_graph(self._h, gid, arr, len(layers)))
        self.load_params(gid, layers, params)

    def load_params(self, gid, layers, params):
        """utils.restore_params equivalent (utils/utils.py:84-93) from a name -> array mapping."""
        for i, l in enumerate(layers):
            try:
                k = np.ascontiguousarray(params[l.scope + "/kernel"], dtype=np.float32)
                b = np.ascontiguousarray(params[l.scope + "/bias"], dtype=np.float32)
            except KeyError as e:
                raise KeyError(f"checkpoint has no variable {e.args[0]!r}") from None
            if k.shape != l.kernel_shape or b.shape != (l.cout,):
                raise ValueError(f"{l.scope}: kernel {k.shape} / bias {b.shape}, expected {l.kernel_shape} / ({l.cout},)")
            self._check(self.lib.tic_load_weights(self._h, gid, i, k.ctypes.data, b.ctypes.data))

    def set_postfilter(self, params=None, mean=None, std=None, name="rmbe", seed=4321):
        """rmbe_model.model graph + 'rmbe/rmbe_params/params' + 'rmbe/channel_normalization_params.npz'
        (submit/2/rmbe/rmbe.py:40-44, submit/2/rmbe/model.py:26-29)."""
        self.post_layers = V.postfilter_layers(name)
        self._set_graph(L.GRAPH_POSTFILTER, self.post_layers,
                        params if params is not None else reference_init(self.post_layers, seed))
        m = np.asarray(self.mean if mean is None else mean, dtype=np.float32).reshape(3)
        s = np.asarray(self.std if std is None else std, dtype=np.float32).reshape(3)
        self.post_mean, self.post_std = m, s
        self._check(self.lib.tic_set_norm(self._h, L.GRAPH_POSTFILTER, m.ctypes.data, s.ctypes.data))

    def set_compute(self, mode):
        m = {"fp32": L.COMPUTE_FP32, "tensor": L.COMPUTE_TENSOR_F16X3, "f16x3": L.COMPUTE_TENSOR_F16X3,
             "3xtf32": L.COMPUTE_TENSOR_3XTF32, "tf32": L.COMPUTE_TENSOR_TF32}[mode] if isinstance(mode, str) else int(mode)
        self._check(self.lib.tic_set_compute_mode(self._h, m))
        self.compute = mode

    def set_chunk_patches(self, chunk):
        self._check(self.lib.tic_set_chunk_patches(self._h, int(chunk)))

    def _follow_torch_stream(self):
        """Device-tensor calls are asynchronous on torch's CURRENT stream (like any torch op), so later
        torch work on that stream — .cpu(), comparisons, NCCL — is ordered after the codec's kernels."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        if getattr(self, "_stream", None) != s:
            self._check(self.lib.tic_set_stream(self._h, C.c_void_p(s)))
            self._stream = s

    def use_torch_stream(self, stream=None):
        """Run on a torch CUDA stream (default: torch's current stream) so torch ops and events order
        against the codec's kernels."""
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self.lib.tic_set_stream(self._h, C.c_void_p(s.cuda_stream)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.tic_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- shapes --------------------------------------------------------------------------------
    def bottleneck_shape(self, patch_size):
        hb, wb, cb = C.c_int(), C.c_int(), C.c_int()
        self._check(self.lib.tic_bottleneck_shape(self._h, int(patch_size), C.byref(hb), C.byref(wb), C.byref(cb)))
        return hb.value, wb.value, cb.value

    @staticmethod
    def _expect_shape(what, x, shape):
        """The C side reads / writes exactly prod(shape) elements: a wrong-sized caller buffer must be a ValueError
        here, never an out-of-bounds access there."""
        if tuple(int(v) for v in x.shape) != tuple(int(v) for v in shape):
            raise ValueError(f"{what} must have shape {tuple(shape)}, got {tuple(x.shape)}")

    def _alloc_like(self, ref, shape, dtype):
        if _is_torch(ref):
            tdt = {np.uint8: torch.uint8, np.float32: torch.float32}[dtype]
            return torch.empty(shape, dtype=tdt, device=ref.device)
        return np.empty(shape, dtype=dtype)

    # ---- hot path ------------------------------------------------------------------------------
    def encode_patches(self, patches, out=None, out_dtype=np.uint8):
        """model.encoder on [N,P,P,3] uint8/float32 patches -> [N,hb,wb,cb] symbols."""
        n, P = int(patches.shape[0]), int(patches.shape[1])
        if tuple(patches.shape[1:]) != (P, P, 3):
            raise ValueError(f"patches must be [N,P,P,3], got {tuple(patches.shape)}")
        in_dt = np.uint8 if str(patches.dtype).endswith("uint8") else np.float32
        src = _Buf(patches, in_dt, self.device, self)
        hb, wb, cb = self.bottleneck_shape(P)
        if out is None:
            out = self._alloc_like(patches, (n, hb, wb, cb), out_dtype)
        else:
            out_dtype = np.uint8 if str(out.dtype).endswith("uint8") else np.float32
            self._expect_shape("out", out, (n, hb, wb, cb))
        dst = _Buf(out, out_dtype, self.device)
        if dst.mem != src.mem:
            raise ValueError("input and output must both be host or both be device buffers")
        self._check(self.lib.tic_encode_patches(self._h, src.ptr, L.U8 if in_dt == np.uint8 else L.F32, n, P, dst.ptr,
                                                L.U8 if out_dtype == np.uint8 else L.F32, src.mem))
        return out

    def encode_images(self, images, patch_size, out=None):
        """crop_image_input_patches + encoder fused: [B,H,W,3] uint8 -> [B, gh*gw, hb, wb, cb] uint8."""
        if images.ndim == 3:
            images = images[None]
        B, H, W = int(images.shape[0]), int(images.shape[1]), int(images.shape[2])
        src = _Buf(images, np.uint8, self.device, self)
        P = int(patch_size)
        hb, wb, cb = self.bottleneck_shape(P)
        gh, gw = -(-H // P), -(-W // P)
        if tuple(images.shape[3:]) != (3,):
            raise ValueError(f"images must be [B,H,W,3], got {tuple(images.shape)}")
        if out is None:
            out = self._alloc_like(images, (B, gh * gw, hb, wb, cb), np.uint8)
        else:
            self._expect_shape("out", out, (B, gh * gw, hb, wb, cb))
        dst = _Buf(out, np.uint8, self.device)
        if dst.mem != src.mem:
            raise ValueError("input and output must both be host or both be device buffers")
        self._check(self.lib.tic_encode_images(self._h, src.ptr, B, H, W, P, dst.ptr, src.mem))
        return out

    def decode_patches(self, symbols, out=None):
        """model.decoder on [N,hb,wb,cb] uint8 symbols -> [N,P,P,3] float32 in [0,255]."""
        n, hb, wb, cb = (int(v) for v in symbols.shape)
        if cb != self.dec_layers[0].cin:
            raise ValueError(f"decoder expects {self.dec_layers[0].cin} symbol channels, got {cb}")
        src = _Buf(symbols, np.uint8, self.device, self)
        up = 2 ** sum(1 for l in self.dec_layers if l.kind == "d")
        down = 1
        for l in self.dec_layers:
            if l.kind == "c":
                down *= l.stride
        P = hb * up // down
        if hb != wb:
            raise ValueError(f"symbol maps must be square, got {hb}x{wb}")
        if out is None:
            out = self._alloc_like(symbols, (n, P, P, 3), np.float32)
        else:
            self._expect_shape("out", out, (n, P, P, 3))
        dst = _Buf(out, np.float32, self.device)
        if dst.mem != src.mem:
            raise ValueError("input and output must both be host or both be device buffers")
        self._check(self.lib.tic_decode_patches(self._h, src.ptr, n, hb, wb, dst.ptr, src.mem))
        return out

    def decode_images(self, symbols, height, width, patch_size, out=None, out_dtype=np.uint8):
        """decoder + concat_patches (+ np.around -> uint8) fused: symbols [B, gh*gw, hb, wb, cb] uint8 ->
        [B,H,W,3] uint8 (rounded) or float32."""
        B = int(symbols.shape[0])
        gh, gw = -(-int(height) // int(patch_size)), -(-int(width) // int(patch_size))
        # exactly the bottleneck shape this variant produces for this patch size (the C side reads
        # gh*gw*hb*wb*cb bytes per image unconditionally: files of another variant / patch size must fail here)
        hb, wb, cb = self.bottleneck_shape(int(patch_size))
        if cb != self.dec_layers[0].cin:
            raise ValueError(f"decoder expects {self.dec_layers[0].cin} symbol channels, the encoder graph produces {cb}")
        self._expect_shape("symbols", symbols, (B, gh * gw, hb, wb, cb))
        src = _Buf(symbols, np.uint8, self.device, self)
        if out is None:
            out = self._alloc_like(symbols, (B, int(height), int(width), 3), out_dtype)
        else:
            out_dtype = np.uint8 if str(out.dtype).endswith("uint8") else np.float32
            self._expect_shape("out", out, (B, int(height), int(width), 3))
        dst = _Buf(out, out_dtype, self.device)
        if dst.mem != src.mem:
            raise ValueError("input and output must both be host or both be device buffers")
        self._check(self.lib.tic_decode_images(self._h, src.ptr, B, int(height), int(width), int(patch_size), dst.ptr,
                                               L.U8 if out_dtype == np.uint8 else L.F32, src.mem))
        return out

    def roundtrip_images(self, images, patch_size, out=None, out_symbols=None, out_dtype=np.uint8, want_symbols=True):
        """test.py:95-146 (compress_and_uncompress): encoder -> decoder in one call, [B,H,W,3] uint8 ->
        (reconstruction [B,H,W,3] uint8 | float32, symbols [B, gh*gw, hb, wb, cb] uint8 | None).  Identical
        results to encode_images + decode_images; host buffers stream through both PCIe directions at once."""
        if images.ndim == 3:
            images = images[None]
        B, H, W = int(images.shape[0]), int(images.shape[1]), int(images.shape[2])
        src = _Buf(images, np.uint8, self.device, self)
        P = int(patch_size)
        hb, wb, cb = self.bottleneck_shape(P)
        gh, gw = -(-H // P), -(-W // P)
        if tuple(images.shape[3:]) != (3,):
            raise ValueError(f"images must be [B,H,W,3], got {tuple(images.shape)}")
        if out is None:
            out = self._alloc_like(images, (B, H, W, 3), out_dtype)
        else:
            out_dtype = np.uint8 if str(out.dtype).endswith("uint8") else np.float32
            self._expect_shape("out", out, (B, H, W, 3))
        dst = _Buf(out, out_dtype, self.device)
        if out_symbols is None and (want_symbols or src.mem == L.MEM_DEVICE):
            out_symbols = self._alloc_like(images, (B, gh * gw, hb, wb, cb), np.uint8)
        elif out_symbols is not None:
            self._expect_shape("out_symbols", out_symbols, (B, gh * gw, hb, wb, cb))
        sym = _Buf(out_symbols, np.uint8, self.device) if out_symbols is not None else None
        if dst.mem != src.mem or (sym is not None and sym.mem != src.mem):
            raise ValueError("input and outputs must all be host or all be device buffers")
        self._check(self.lib.tic_roundtrip_images(self._h, src.ptr, B, H, W, P, sym.ptr if sym is not None else None,
                                                  dst.ptr, L.U8 if out_dtype == np.uint8 else L.F32, src.mem))
        return out, out_symbols

    def postfilter_patches(self, tiles, out=None):
        """rmbe_model.model on [N,P,P,3] float32 tiles."""
        if self.post_layers is None:
            raise TicError("post-filter not configured (set_postfilter)")
        n, P = int(tiles.shape[0]), int(tiles.shape[1])
        if tuple(tiles.shape[1:]) != (P, P, 3):
            raise ValueError(f"tiles must be [N,P,P,3], got {tuple(tiles.shape)}")
        src = _Buf(tiles, np.float32, self.device, self)
        if out is None:
            out = self._alloc_like(tiles, tuple(tiles.shape), np.float32)
        else:
            self._expect_shape("out", out, tuple(tiles.shape))
        dst = _Buf(out, np.float32, self.device)
        self._check(self.lib.tic_postfilter_patches(self._h, src.ptr, n, P, dst.ptr, src.mem))
        return out

    def postfilter_images(self, images):
        """rmbe.rmbe in place over float32 [B,H,W,3] (or [H,W,3]) images."""
        if self.post_layers is None:
            raise TicError("post-filter not configured (set_postfilter)")
        # the C side reads and writes H*W*3 floats per image: any other layout must fail here
        if images.ndim not in (3, 4) or tuple(images.shape[-1:]) != (3,):
            raise ValueError(f"images must be [B,H,W,3] or [H,W,3], got {tuple(images.shape)}")
        x = images if images.ndim == 4 else images[None]
        B, H, W = int(x.shape[0]), int(x.shape[1]), int(x.shape[2])
        buf = _Buf(x, np.float32, self.device, self)
        self._check(self.lib.tic_postfilter_images(self._h, buf.ptr, B, H, W, buf.mem))
        return images

    def run_layers(self, graph, x, n_layers):
        """Layers [0, n_layers) of 'encoder' | 'decoder' | 'postfilter' on f32 NHWC activations (no fused
        prologue / epilogue): the tensor a sess.run on an intermediate op would return."""
        gid = {"encoder": L.GRAPH_ENCODER, "decoder": L.GRAPH_DECODER, "postfilter": L.GRAPH_POSTFILTER}[graph]
        layers = {"encoder": self.enc_layers, "decoder": self.dec_layers, "postfilter": self.post_layers}[graph]
        n, h0, w0, _ = (int(v) for v in x.shape)
        h, w = h0, w0
        for l in layers[:n_layers]:
            h, w = ((-(-h // l.stride), -(-w // l.stride)) if l.kind == "c" else (2 * h, 2 * w))
        src = _Buf(x, np.float32, self.device, self)
        out = self._alloc_like(x, (n, h, w, layers[n_layers - 1].cout), np.float32)
        dst = _Buf(out, np.float32, self.device)
        self._check(self.lib.tic_run_layers(self._h, gid, src.ptr, n, h0, w0, int(n_layers), dst.ptr, src.mem))
        return out

    def round_u8(self, x, out=None):
        src = _Buf(x, np.float32, self.device, self)
        if out is None:
            out = self._alloc_like(x, tuple(x.shape), np.uint8)
        else:
            self._expect_shape("out", out, tuple(x.shape))
        dst = _Buf(out, np.uint8, self.device)
        n = int(np.prod(x.shape))
        self._check(self.lib.tic_round_u8(self._h, src.ptr, dst.ptr, n, src.mem))
        return out

    # ---- statistics ----------------------------------------------------------------------------
    def hist_reset(self):
        self._check(self.lib.tic_hist_reset(self._h))

    def hist_read(self):
        """freq[q] of every symbol encoded since the last reset (get_encoded_distribution.py:113-126)."""
        counts = np.zeros(self.quan_scale, dtype=np.uint64)
        self._check(self.lib.tic_hist_read(self._h, counts.ctypes.data, self.quan_scale))
        return counts

    def hist_device_ptr(self):
        p = C.c_void_p()
        self._check(self.lib.tic_hist_device_ptr(self._h, C.byref(p)))
        return p.value

    def position_sums(self, symbols, sums=None):
        """sums[hb*wb*cb] += sum over patches (cal_encoded_distribution.py:111-128)."""
        n = int(symbols.shape[0])
        npos = int(np.prod(symbols.shape[1:]))
        src = _Buf(symbols, np.uint8, self.device, self)
        if sums is None:
            sums = (torch.zeros(npos, dtype=torch.int64, device=symbols.device) if _is_torch(symbols)
                    else np.zeros(npos, dtype=np.uint64))
        ptr = sums.data_ptr() if _is_torch(sums) else sums.ctypes.data
        self._check(self.lib.tic_position_sums(self._h, src.ptr, n, npos, ptr, src.mem))
        return sums

    def position_sums_batched(self, symbols, batch=64):
        """Exact per-batch integer sums [ceil(n/batch), hb*wb*cb] (uint64): what one sess.run batch contributes to the
        reference's running mean (cal_encoded_distribution.py:111-128, batch_size = 64 at :92)."""
        n = int(symbols.shape[0])
        npos = int(np.prod(symbols.shape[1:]))
        nb = -(-n // int(batch))
        src = _Buf(symbols, np.uint8, self.device, self)
        sums = (torch.zeros((nb, npos), dtype=torch.int64, device=symbols.device) if _is_torch(symbols)
                else np.zeros((nb, npos), dtype=np.uint64))
        if n:
            ptr = sums.data_ptr() if _is_torch(sums) else sums.ctypes.data
            self._check(self.lib.tic_position_sums_batched(self._h, src.ptr, n, npos, int(batch), ptr, src.mem))
        return sums

    # ---- GPU entropy stage ----------------------------------------------------------------------
    def entropy_bound(self, stream_len):
        return int(self.lib.tic_entropy_bound(int(stream_len)))

    def entropy_encode(self, symbols, cum_freq):
        """encode.py:171-202 on the device: symbols [n_streams, ...] uint8 (one image's patch-major symbol sequence per
        row, e.g. the result of encode_images) -> (out uint8 [n_streams, bound], nbytes int64 [n_streams]); stream i is
        out[i, :nbytes[i]], byte-identical to range_coder.RangeEncoder(path).encode(symbols[i].reshape(-1), cum_freq);
        close().  Device tensors stay on the device (asynchronous; errors surface through check_status())."""
        n = int(symbols.shape[0])
        slen = int(np.prod(symbols.shape[1:])) if n else 0
        src = _Buf(symbols, np.uint8, self.device, self)
        cum = np.ascontiguousarray(np.asarray([int(v) for v in cum_freq], dtype=np.uint32))
        stride = self.entropy_bound(slen)
        out = self._alloc_like(symbols, (n, stride), np.uint8)
        nbytes = (torch.zeros(n, dtype=torch.int64, device=symbols.device) if _is_torch(symbols) else np.zeros(n, dtype=np.int64))
        dst = _Buf(out, np.uint8, self.device)
        nb_ptr = nbytes.data_ptr() if _is_torch(nbytes) else nbytes.ctypes.data
        self._check(self.lib.tic_entropy_encode(self._h, src.ptr, n, slen, cum.ctypes.data, cum.size, dst.ptr, stride, nb_ptr, src.mem))
        return out, nbytes

    def entropy_decode(self, streams, nbytes, stream_len, cum_freq, out=None):
        """decode.py:79-101,182 on the device: streams uint8 [n_streams, stride] (stride a multiple of 16) holding
        nbytes[i] stored bytes each -> symbols uint8 [n_streams, stream_len]."""
        n, stride = int(streams.shape[0]), int(streams.shape[1])
        src = _Buf(streams, np.uint8, self.device, self)
        cum = np.ascontiguousarray(np.asarray([int(v) for v in cum_freq], dtype=np.uint32))
        if _is_torch(streams):
            nb = nbytes.to(device=streams.device, dtype=torch.int64).contiguous()
            nb_ptr = nb.data_ptr()
        else:
            nb = np.ascontiguousarray(np.asarray(nbytes, dtype=np.int64))
            nb_ptr = nb.ctypes.data
        if int(nb.shape[0]) != n:
            raise ValueError("nbytes must have one entry per stream")
        if out is None:
            out = self._alloc_like(streams, (n, int(stream_len)), np.uint8)
        else:
            self._expect_shape("out", out.reshape(n, -1) if n else out, (n, int(stream_len)))
        dst = _Buf(out, np.uint8, self.device)
        if dst.mem != src.mem:
            raise ValueError("input and output must both be host or both be device buffers")
        self._check(self.lib.tic_entropy_decode(self._h, src.ptr, n, stride, nb_ptr, cum.ctypes.data, cum.size, dst.ptr,
                                                int(stream_len), src.mem))
        return out

    # ---- rate-distortion evaluation -------------------------------------------------------------
    def evaluate_images(self, images, patch_size, cum_freq, out=None):
        """encode.py -> decode.py -> processing_utils/evaluate.py on the device, without files: [B,H,W,3] uint8 ->
        (code_bytes int64[B], sq_err uint64[B], out | None).  code_bytes[i] is the size of the range-coded file of image i
        (entropy_encode's nbytes, entry.compress's file), sq_err[i] the integer sum of squared differences between image i
        and its uint8 reconstruction (decode_images), written to `out` [B,H,W,3] uint8 when one is given.  CUDA tensors in
        give CUDA tensors out (sq_err as int64; asynchronous, errors surface through check_status())."""
        if images.ndim == 3:
            images = images[None]
        B, H, W = int(images.shape[0]), int(images.shape[1]), int(images.shape[2])
        if tuple(images.shape[3:]) != (3,):
            raise ValueError(f"images must be [B,H,W,3], got {tuple(images.shape)}")
        src = _Buf(images, np.uint8, self.device, self)
        cum = np.ascontiguousarray(np.asarray([int(v) for v in cum_freq], dtype=np.uint32))
        dst = None
        if out is not None:
            self._expect_shape("out", out, (B, H, W, 3))
            dst = _Buf(out, np.uint8, self.device)
            if dst.mem != src.mem:
                raise ValueError("input and output must both be host or both be device buffers")
        if _is_torch(images) and images.is_cuda:
            code_bytes = torch.zeros(B, dtype=torch.int64, device=images.device)
            sq_err = torch.zeros(B, dtype=torch.int64, device=images.device)
            cb_ptr, se_ptr = code_bytes.data_ptr(), sq_err.data_ptr()
        else:
            code_bytes, sq_err = np.zeros(B, dtype=np.int64), np.zeros(B, dtype=np.uint64)
            cb_ptr, se_ptr = code_bytes.ctypes.data, sq_err.ctypes.data
        self._check(self.lib.tic_evaluate_images(self._h, src.ptr, B, H, W, int(patch_size), cum.ctypes.data, cum.size, cb_ptr,
                                                 se_ptr, dst.ptr if dst is not None else None, src.mem))
        return code_bytes, sq_err, out

    def check_status(self):
        """Synchronise the codec's stream and raise if a tensor-mode ('f16x3') run left the fp16 range (|activation| >=
        65504): device-buffer calls are asynchronous, so their status surfaces here or at the next call."""
        self._check(self.lib.tic_check_status(self._h))

    # ---- measurement ---------------------------------------------------------------------------
    @property
    def launch_count(self):
        return int(self.lib.tic_launch_count(self._h))

    def profile(self, on=True):
        """Bracket every layer launch with CUDA events (per-layer device times, see layer_times)."""
        self._check(self.lib.tic_profile_enable(self._h, int(bool(on))))
        self._check(self.lib.tic_profile_reset(self._h))

    def layer_times(self, graph):
        """[(scope, total_ms, launches)] per primitive layer of 'encoder' | 'decoder' | 'postfilter'
        accumulated since profile(True)."""
        gid = {"encoder": L.GRAPH_ENCODER, "decoder": L.GRAPH_DECODER, "postfilter": L.GRAPH_POSTFILTER}[graph]
        layers = {"encoder": self.enc_layers, "decoder": self.dec_layers, "postfilter": self.post_layers}[graph]
        ms = np.zeros(len(layers), dtype=np.float32)
        cnt = np.zeros(len(layers), dtype=np.int64)
        self._check(self.lib.tic_profile_read(self._h, gid, ms.ctypes.data, cnt.ctypes.data, len(layers)))
        return [(l, float(m), int(c)) for l, m, c in zip(layers, ms, cnt)]

    def last_kernel_ms(self):
        return float(self.lib.tic_last_kernel_ms(self._h))
