"""TEST INFRASTRUCTURE: the Codec's public surface implemented with the CPU oracle, so that the host-side product
logic above the C ABI (entry.py, model_api.py, compat.py, range_coder.py, checkpoint.py) can be driven where no GPU is
present — in particular by the reference's unmodified encode.py / decode.py (tests/test_dropin.py)."""
import numpy as np

from oracle import codec_oracle as O
from tf_image_compression_b200 import variants as V


class OracleCodec:
    def __init__(self, variant, quan_scale, mean, std, enc_params, dec_params, post_params=None, post_mean=None,
                 post_std=None, post_name="rmbe"):
        self.variant = V.resolve(variant)
        self.quan_scale = int(quan_scale)
        self.mean, self.std = np.asarray(mean, np.float32), np.asarray(std, np.float32)
        self.enc_params, self.dec_params = dict(enc_params), dict(dec_params)
        self.enc_layers = V.encoder_layers(self.variant)
        self.dec_layers = V.decoder_layers(self.variant)
        self.device = 0
        self.calls = []
        # the rmbe post-filter of submit/2 (Codec.set_postfilter): weights, normalisation and net
        self.post_params = None if post_params is None else dict(post_params)
        self.post_mean = self.mean if post_mean is None else np.asarray(post_mean, np.float32)
        self.post_std = self.std if post_std is None else np.asarray(post_std, np.float32)
        self.post_name = post_name

    # ---- Codec surface used by ModelModule / entry / checkpoint ------------------------------------------------
    def bottleneck_shape(self, patch_size):
        h = int(patch_size)
        for l in self.enc_layers:
            h = -(-h // l.stride) if l.kind == "c" else 2 * h
        return h, h, self.enc_layers[-1].cout

    def load_params(self, gid, layers, params):
        dst = self.enc_params if layers is self.enc_layers else self.dec_params
        for l in layers:
            for s in ("/kernel", "/bias"):
                dst[l.scope + s] = np.asarray(params[l.scope + s], np.float32)

    def encode_patches(self, patches, out=None, out_dtype=np.uint8):
        self.calls.append(("encode_patches", len(patches)))
        sym = O.encoder(np.asarray(patches, np.float32), self.variant, self.enc_params, self.mean, self.std, self.quan_scale)
        return sym.astype(out_dtype)

    def decode_patches(self, symbols, out=None):
        self.calls.append(("decode_patches", len(symbols)))
        return O.decoder(np.asarray(symbols), self.variant, self.dec_params, self.mean, self.std, self.quan_scale)

    def encode_images(self, images, patch_size, out=None):
        out = []
        for im in np.asarray(images):
            p = np.stack(O.crop_image_input_patches(im, patch_size)).astype(np.float32)
            out.append(O.encoder(p, self.variant, self.enc_params, self.mean, self.std, self.quan_scale))
        return np.stack(out)

    def decode_images(self, symbols, height, width, patch_size, out=None, out_dtype=np.uint8):
        out = []
        for s in np.asarray(symbols):
            rec = O.decoder(s, self.variant, self.dec_params, self.mean, self.std, self.quan_scale)
            img = O.concat_patches(list(rec), height, width, patch_size)
            out.append(O.around_u8(img) if out_dtype == np.uint8 else img.astype(np.float32))
        return np.stack(out)

    def postfilter_images(self, images):
        """O.rmbe in place over float32 [B,H,W,3] (or [H,W,3]) images."""
        if self.post_params is None:
            raise RuntimeError("post-filter not configured")
        x = images if images.ndim == 4 else images[None]
        for im in x:
            im[...] = O.rmbe(im, lambda t: O.postfilter(t, self.post_name, self.post_params, self.post_mean, self.post_std))
        return images

    def round_u8(self, x, out=None):
        return O.around_u8(np.asarray(x))
