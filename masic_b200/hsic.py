"""HSIC — MASIC's stereo codec model on the B200-native engine.

Same public surface as the reference's `HSIC(CompressionModel)`
(coremasic/mywork/MASIC.py:40-110, 652-851): constructor `HSIC(N=128, M=192, K=5)`,
`forward(x1, x2, h_matrix) -> dict`, `update(force)`, `aux_loss()`, `parameters()` /
`aux_parameters()` split, and a `state_dict()` with the reference's 248 entries (names,
shapes, dtypes), so checkpoints move both ways.  Parameters are created in the reference's
order with the same initialisers, hence `torch.manual_seed(s); HSIC()` draws the same
weights as the reference.

`forward` does not execute the module tree: it hands the state_dict to an `HSICEngine`
(masic_b200/engine.py) compiled for the input's (batch, H, W) and replays its CUDA graph.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import ops as _ops
from ._lib import MasicError
from .engine import HSICEngine
from .entropy_models import EntropyBottleneck, GaussianMixtureConditional_gf
from .layers import GDN, MaskedConv2d, conv, deconv
from .padding import padding_for, run_engine


class _Block(nn.Module):
    """Parameter container (the engine, not the module tree, executes the forward pass)."""


def _encoder(N: int, M: int, second_view: bool) -> nn.Module:
    b = _Block()
    if second_view:                       # MASIC.py:559-560
        b.pre_conv = conv(6, 3, stride=1)
        b.pre_gdn = GDN(3)
    b.g_a_conv1 = conv(3, N)              # MASIC.py:513-519 / :562-568
    b.g_a_gdn1 = GDN(N)
    b.g_a_conv2 = conv(N, N)
    b.g_a_gdn2 = GDN(N)
    b.g_a_conv3 = conv(N, N)
    b.g_a_gdn3 = GDN(N)
    b.g_a_conv4 = conv(N, M)
    return b


def _decoder(N: int, M: int, second_view: bool) -> nn.Module:
    b = _Block()
    b.g_s_conv1 = deconv(M, N)            # MASIC.py:536-542 / :590-596
    b.g_s_gdn1 = GDN(N, inverse=True)
    b.g_s_conv2 = deconv(N, N)
    b.g_s_gdn2 = GDN(N, inverse=True)
    b.g_s_conv3 = deconv(N, N)
    b.g_s_gdn3 = GDN(N, inverse=True)
    b.g_s_conv4 = deconv(N, 3)
    if second_view:                       # MASIC.py:599-600
        b.after_gdn = GDN(3, inverse=True)
        b.after_conv = deconv(6, 3, stride=1)
    return b


def _hyper_analysis(N: int, M: int) -> nn.Module:
    b = _Block()                          # MASIC.py:170-183
    b.encode_hyper = nn.Sequential(conv(M, N, kernel_size=5, stride=1), nn.ReLU(inplace=True),
                                   conv(N, N, kernel_size=5), nn.ReLU(inplace=True), conv(N, N, kernel_size=5))
    return b


def _hyper_synthesis_up(N: int, M: int) -> nn.Sequential:
    return nn.Sequential(deconv(N, M, stride=2, kernel_size=5), nn.LeakyReLU(inplace=True),   # MASIC.py:678-691
                         deconv(M, M * 3 // 2, stride=2, kernel_size=5), nn.LeakyReLU(inplace=True),
                         conv(M * 3 // 2, M * 2, stride=1, kernel_size=3))


def _gmm_param_net(N: int, M: int, K: int, c_in: int, transposed_head: bool) -> nn.Module:
    """MASIC.py:330-376 (y1: ConvTranspose2d k=1 for the first two layers) / :399-444 (y2)."""
    head = deconv if transposed_head else conv
    b = _Block()
    b.N, b.M, b.K = N, M, K
    b.gmm_sigma = nn.Sequential(head(c_in, 6 * M, kernel_size=1, stride=1), nn.ReLU(inplace=True),
                                head(6 * M, 4 * M, kernel_size=1, stride=1), nn.ReLU(inplace=True),
                                conv(4 * M, M * K, kernel_size=1, stride=1), nn.ReLU(inplace=True))
    b.gmm_means = nn.Sequential(head(c_in, 6 * M, kernel_size=1, stride=1), nn.LeakyReLU(inplace=True),
                                head(6 * M, 4 * M, kernel_size=1, stride=1), nn.LeakyReLU(inplace=True),
                                conv(4 * M, M * K, kernel_size=1, stride=1))
    b.gmm_weights = nn.Sequential(head(c_in, 6 * M, kernel_size=1, stride=1), nn.LeakyReLU(inplace=True),
                                  head(6 * M, M * K, kernel_size=1, stride=1), nn.LeakyReLU(inplace=True),
                                  conv(M * K, M * K, kernel_size=1, stride=1))
    return b


def _mask2weights(Kw: int = 3) -> nn.Module:
    b = _Block()                          # MASIC.py:472-491
    b.maskconv = nn.Sequential(conv(1, 3, kernel_size=3, stride=2), nn.ReLU(inplace=True),
                               conv(3, 6, kernel_size=3), nn.ReLU(inplace=True),
                               conv(6, 6, kernel_size=3), nn.ReLU(inplace=True), conv(6, 3, kernel_size=3))
    b.Kw = Kw
    return b


class HSIC(nn.Module):
    def __init__(self, N: int = 128, M: int = 192, K: int = 5, use_cuda_graph: bool = True, **kwargs):
        super().__init__()
        self.entropy_bottleneck1 = EntropyBottleneck(N)          # MASIC.py:50-54
        self.entropy_bottleneck2 = EntropyBottleneck(N)
        self.gaussian1 = GaussianMixtureConditional_gf(K=K)      # :658-659
        self.gaussian2 = GaussianMixtureConditional_gf(K=K)
        self.N, self.M, self.K = int(N), int(M), int(K)
        self.encoder1 = _encoder(N, M, False)                    # :664-667
        self.encoder2 = _encoder(N, M, True)
        self.decoder1 = _decoder(N, M, False)
        self.decoder2 = _decoder(N, M, True)
        self._h_a1 = _hyper_analysis(N, M)                       # :672-673
        self._h_a2 = _hyper_analysis(N, M)
        self.h_s1_up = _hyper_synthesis_up(N, M)                 # :678-691
        self.h_s2_up = _hyper_synthesis_up(N, M)
        self.context_prediction1 = MaskedConv2d(M, 2 * M, kernel_size=5, padding=2, stride=1)   # :693-703
        self.context_prediction2 = MaskedConv2d(M, 2 * M, kernel_size=5, padding=2, stride=1)
        self._h_s1_same_resolution = _gmm_param_net(N, M, K, 4 * M, True)                         # :704-705
        self._h_s2_same_resolution = _gmm_param_net(N, M, K, 5 * M, False)
        self.mask2weights_unit = _mask2weights(3)                # :706
        self._use_graph = use_cuda_graph
        self._engines: Dict[Tuple, HSICEngine] = {}
        self._engine_version = 0
        self._staging_key, self._staging = None, {}

    # ---- CompressionModel surface (MASIC.py:59-109)
    def aux_loss(self):
        return sum(m.loss() for m in self.modules() if isinstance(m, EntropyBottleneck))

    def parameters(self, recurse: bool = True):
        for m in self.children():
            if isinstance(m, EntropyBottleneck):
                continue
            for p in m.parameters():
                yield p

    def aux_parameters(self):
        for m in self.children():
            if not isinstance(m, EntropyBottleneck):
                continue
            for p in m.parameters():
                yield p

    def update(self, force: bool = False):
        for m in self.children():
            if isinstance(m, EntropyBottleneck):
                m.update(force=force)

    # ---- engine management
    def _weights_fingerprint(self):
        return tuple(p._version for p in nn.Module.parameters(self))

    def invalidate_engines(self):
        """Call after mutating weights in place (load_state_dict does it automatically)."""
        self._engines.clear()

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        # CDF buffers are empty (0,) tensors in checkpoints until update() (SURVEY §5): resize to fit
        for name in ("entropy_bottleneck1", "entropy_bottleneck2", "gaussian1", "gaussian2"):
            mod = getattr(self, name)
            for buf in ("_offset", "_quantized_cdf", "_cdf_length", "scale_table"):
                key = f"{name}.{buf}"
                if key in state_dict and hasattr(mod, buf):
                    cur = getattr(mod, buf)
                    if cur.shape != state_dict[key].shape:
                        setattr(mod, buf, torch.empty(state_dict[key].shape, dtype=cur.dtype, device=cur.device))
        res = super().load_state_dict(state_dict, strict=strict, **kw)
        self.invalidate_engines()
        return res

    def engine_for(self, batch: int, height: int, width: int, device) -> HSICEngine:
        key = (batch, height, width, str(device), self._weights_fingerprint())
        eng = self._engines.get(key)
        if eng is None:
            self._engines.clear()
            # MaskedConv2d side effect of the reference's forward (layers.py:77): weight.data *= mask
            with torch.no_grad():
                for cp in (self.context_prediction1, self.context_prediction2):
                    cp.weight.data *= cp.mask
            key = (batch, height, width, str(device), self._weights_fingerprint())
            eng = HSICEngine(self.state_dict(), batch, height, width, device, self.N, self.M, self.K,
                             use_graph=self._use_graph)
            self._engines[key] = eng
        return eng

    # ---- forward (MASIC.py:744-851)
    def forward(self, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor, clone: bool = True):
        """MASIC.py:744-851 at any H, W: a pair whose size is not a multiple of 64 runs zero-padded on the device, as
        CompressAI evaluates it (masic_b200/padding.py); x1_hat, x2_hat and the masks are cropped back to (H, W), the
        latents and likelihoods stay on the padded grid."""
        if self.training:
            raise MasicError("HSIC.forward in train() mode does not build an autograd graph: the training step "
                             "(noise quantisation, loss, backward, aux loss) runs as fused CUDA kernels through "
                             "model.trainer(batch, H, W, device, lmbda).train_step(x1, x2, h, optimizer, aux_optimizer)")
        if not x1.is_cuda:
            raise MasicError("HSIC.forward needs CUDA tensors: masic_b200 has no CPU fallback")
        b, _, h, w = x1.shape
        pad = padding_for(h, w)
        eng = self.engine_for(b, pad.hp, pad.wp, x1.device)
        o = run_engine(eng, pad, x1, x2, h_matrix)
        c = (lambda t: t.clone()) if clone else (lambda t: t)
        if not pad.aligned:         # the images cropped back to (h, w); latents and likelihoods stay on the padded grid
            o = {**o, **self._crop(eng, pad, o)}
        return {
            "x1_hat": c(o["x1_hat"]), "x2_hat": c(o["x2_hat"]),
            "y1_hat": c(o["y1_hat"]), "z1_hat": c(o["z1_hat"]),
            "x1_mask_R": c(o["x1_mask_R"]), "x1_mask_L": c(o["x1_mask_L"]),
            "likelihoods": {"y1": c(o["lik_y1"]), "y2": c(o["lik_y2"]), "z1": c(o["lik_z1"]), "z2": c(o["lik_z2"])},
        }

    _CROPPED = ("x1_hat", "x2_hat", "x1_mask_R", "x1_mask_L")

    def _crop(self, eng: HSICEngine, pad, o) -> Dict[str, torch.Tensor]:
        """The padded engine's images cropped to the pair's size, into staging buffers cached per (batch, h, w)."""
        key = (eng.B, pad.h, pad.w, str(eng.dev))
        if self._staging_key != key:
            self._staging_key = key
            self._staging = {k: torch.empty(eng.B, o[k].shape[1], pad.h, pad.w, device=eng.dev) for k in self._CROPPED}
        with torch.cuda.device(eng.dev):
            for k in self._CROPPED:
                pad.crop_into(o[k], self._staging[k])
        return self._staging

    # ---- the same forward, layer by layer (what the unmodified MASIC.py does on masic_b200/compat)
    @torch.no_grad()
    def forward_modules(self, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor):
        """MASIC.py:744-851 (eval) in the reference's own call order, every step one `nn.Module.forward` of
        masic_b200.layers / entropy_models / kornia_compat on NCHW fp32 tensors — the path the reference's model file
        takes when its `compressai` / `kornia` imports resolve to masic_b200/compat (INTEGRATION.md, path B).  No
        engine, no fusion, no CUDA graph: each conv packs its input to NHWC bf16, runs the tensor-core kernel and
        unpacks; GDN, warp, likelihoods are their stand-alone kernels."""
        from . import kornia_compat as kornia
        if self.training:
            raise MasicError("forward_modules implements eval mode (use model.trainer(...) for the training step)")

        def enc(e, x):                                      # Encoder1/2.forward, MASIC.py:521-531 / :570-585
            x = e.g_a_gdn1(e.g_a_conv1(x))
            x = e.g_a_gdn2(e.g_a_conv2(x))
            x = e.g_a_gdn3(e.g_a_conv3(x))
            return e.g_a_conv4(x)

        def dec(d, y):                                      # Decoder1/2.forward, MASIC.py:544-554 / :602-616
            y = d.g_s_gdn1(d.g_s_conv1(y))
            y = d.g_s_gdn2(d.g_s_conv2(y))
            y = d.g_s_gdn3(d.g_s_conv3(y))
            return d.g_s_conv4(y)

        def gmm(net, x):                                    # MASIC.py:378-396 / :446-468
            sigma, mu, lw = net.gmm_sigma(x), net.gmm_means(x), net.gmm_weights(x)
            t = lw.reshape(-1, self.K, self.M, x.shape[-2], x.shape[-1])
            return sigma, mu, torch.softmax(t, dim=-4).reshape(-1, self.M * self.K, x.shape[-2], x.shape[-1])

        size = (x1.size()[-2], x1.size()[-1])
        y1 = enc(self.encoder1, x1)
        z1 = self._h_a1.encode_hyper(torch.abs(y1))
        z1_hat, z1_lik = self.entropy_bottleneck1(z1)
        params1 = self.h_s1_up(z1_hat)
        y1_hat = self.gaussian1._quantize(y1, "dequantize")
        ctx1 = self.context_prediction1(y1_hat)
        y1_hat, y1_lik = self.gaussian1(y1, *gmm(self._h_s1_same_resolution, torch.cat((params1, ctx1), dim=1)))
        x1_hat = dec(self.decoder1, y1_hat)
        x1_warp = kornia.warp_perspective(x1, h_matrix, size)
        e2 = self.encoder2
        y2 = enc(e2, e2.pre_gdn(e2.pre_conv(torch.cat((x1_warp, x2), dim=-3))))
        z2 = self._h_a2.encode_hyper(torch.abs(y2))
        z2_hat, z2_lik = self.entropy_bottleneck2(z2)
        params2 = self.h_s2_up(z2_hat)
        y2_hat = self.gaussian2._quantize(y2, "dequantize")
        ctx2 = self.context_prediction2(y2_hat)
        ones = torch.ones(x1.shape[0], 1, *size, dtype=x1.dtype, device=x1.device)          # mask(), MASIC.py:627-649
        mask_r = kornia.warp_perspective(ones, h_matrix, size)
        mask_l = kornia.warp_perspective(mask_r, torch.inverse(h_matrix), size)
        o = self.mask2weights_unit.maskconv(mask_r)                                          # MASIC.py:493-506
        mw = torch.softmax(o.reshape(-1, 3, 1, o.shape[-2], o.shape[-1]), dim=-4).reshape(-1, 3, o.shape[-2], o.shape[-1])
        x1_hat_warp = kornia.warp_perspective(x1_hat, h_matrix, size)
        y1w_hat = self.gaussian1._quantize(enc(self.encoder1, x1_hat_warp), "dequantize")
        fused = torch.cat((params2 * mw[:, 0:1], ctx2 * mw[:, 1:2], y1w_hat * mw[:, 2:3]), dim=1)
        y2_hat, y2_lik = self.gaussian2(y2, *gmm(self._h_s2_same_resolution, fused))
        d2 = self.decoder2
        x2_hat = d2.after_conv(torch.cat((d2.after_gdn(dec(d2, y2_hat)), x1_hat_warp), dim=-3))
        return {"x1_hat": x1_hat, "x2_hat": x2_hat, "y1_hat": y1_hat, "z1_hat": z1_hat, "x1_mask_R": mask_r,
                "x1_mask_L": mask_l, "likelihoods": {"y1": y1_lik, "y2": y2_lik, "z1": z1_lik, "z2": z2_lik}}

    def pair_stream(self, height: int, width: int, device, depth: int = 2, lmbda: float = 0.0) -> "PairStream":
        """Pipelined host-to-host evaluation of batch-1 stereo pairs (see PairStream)."""
        return PairStream(self, height, width, device, depth=depth, lmbda=lmbda)

    def trainer(self, batch: int, height: int, width: int, device, lmbda: float = 0.01, metric: str = "mse"):
        """The CUDA training step for this model (forward in train() mode + loss + backward + aux loss):
        `HSICTrainer.step_grads` fills `.grad` of every parameter, `train_step` also all-reduces and steps the
        two optimisers (coremasic/mywork/newtrain_codec_real.py:105-146).  metric: "mse" (the reference's loss) or
        "ms-ssim" (CompressAI's MS-SSIM rate-distortion loss on both views, min(H, W) > 160; see HSICTrainer)."""
        from .trainer import HSICTrainer
        return HSICTrainer(self, batch, height, width, device, lmbda=lmbda, metric=metric)

    # ---- bitstreams (MASIC.py:855-1158, :1161-1408)
    def compress(self, x1, x2, h_matrix, output_name, output_path="", device="cpu", y_order="wavefront_streams"):
        """y_order: "wavefront_streams" (default: positions coded wave by wave, one range-coded stream per non-zero
        channel, decoded entirely on the device), "wavefront" (wave order, a single stream, host range decoder) or
        "raster" (the reference's order, per-position decoder).  See masic_b200/bitstream.py."""
        from .bitstream import compress
        return compress(self, x1, x2, h_matrix, output_name, output_path, device, y_order=y_order)

    def decompress(self, x1, x2, h_matrix, output_name, output_path="", device="cpu"):
        from .bitstream import decompress
        return decompress(self, x1, x2, h_matrix, output_name, output_path,
                          None if device == "cpu" else device)

    def compress_batch(self, x1, x2, h_matrix):
        """Code B pairs of one size at once (B, 3, H, W device tensors; h_matrix (B, 3, 3)).  Returns one dict per pair:
        `header` and `payload`, the bytes `compress` writes to `<name>.npz` / `<name>.bin` for that pair alone, and
        `bpp_real`, `n_symbols`, `y_bits_ideal`.  See masic_b200/bitstream.py."""
        from .bitstream import compress_batch
        return compress_batch(self, x1, x2, h_matrix)

    def decompress_batch(self, items, h_matrix, device=None):
        """Decode a list of (header, payload) byte strings of pairs of one size (format 2) with their (B, 3, 3)
        homographies.  Returns x1_hat, x2_hat, y1_hat, y2_hat, z1_hat, z2_hat, batched in the order of items."""
        from .bitstream import decompress_batch
        return decompress_batch(self, items, h_matrix, device)


class PairStream:
    """Pipelined evaluation of stereo pairs that live in HOST memory (the reference's eval loop,
    coremasic/mywork/test2_real.py:172-252: `d.to(device)` -> `model(d1, d2, h)` -> criterion -> `.item()`).

        ps = model.pair_stream(H, W, device)
        t0 = ps.submit(x1_host, x2_host, h_host)     # pinned (1,3,H,W) fp32 x2, (1,3,3) fp32
        t1 = ps.submit(...)                          # its H2D copy overlaps pair 0's kernels
        bpp, psnr1, psnr2 = ps.result(t0)            # the criterion, read back from the device (32 bytes)
        t2 = ps.submit(..., msssim=True)             # + MS-SSIM of both views, in result(t2)[3]
        ps.attach_lpips(lpips_net)                   # a masic_b200.lpips.LPIPS
        t3 = ps.submit(..., lpips=True)              # + LPIPS of both views, in result(t3)[3]
        ps.attach_enhancement(en)                    # a masic_b200.cqe.Independent_EN: full MASIC (test3_real.py)
        t4 = ps.submit(..., enhance=True, msssim=True, lpips=True)   # every number of the enhanced pair

    `depth` slots (default 2), each with its own engine and stream: the H2D copy of pair i+1 runs on a copy stream
    while pair i replays its engine's CUDA graph, and the kernels of consecutive pairs overlap on the GPU; the
    criterion is one fused reduction pass (masic_rd_metrics) whose 8 floats come back through pinned memory; with
    msssim=True the slot's stream also runs masic_ms_ssim on both views and 6 more floats ride in the same read-back;
    with lpips=True its LPIPS engine compares both views and 2 more floats ride along.  With enhance=True the slot's
    CQE engine replays right after the codec, reading the codec's buffers in place, and everything above measures the
    enhanced pair; a second masic_rd_metrics pass adds the codec's own MSE to the same read-back.
    `outputs()` exposes the engine's output tensors of the LAST submitted pair (valid after `result(ticket)`),
    `enhanced_outputs()` the enhanced pair of the last one submitted with enhance=True.
    H and W need not be multiples of 64: each pair is then zero-padded on the device into an engine of the padded size
    and its reconstructions cropped back (masic_b200/padding.py); every number and image refers to the H x W pair.
    """

    def __init__(self, model: "HSIC", height: int, width: int, device, depth: int = 2, lmbda: float = 0.0):
        import ctypes as C
        from . import _lib
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("PairStream needs a CUDA device: masic_b200 has no CPU fallback")
        self.model, self.H, self.W, self.lmbda = model, height, width, float(lmbda)
        self.depth = depth
        self.pad = pad = padding_for(height, width)
        # One engine (static buffers + CUDA graph) per slot, each replayed on its own stream: the H2D copy lands
        # directly in the engine's input buffers (no staging copy), and the kernels of consecutive pairs overlap —
        # the tail of a pair is a chain of launches that leave SMs idle (conv4: 85 tiles, hyper-prior layers: 10-40),
        # which the next pair's kernels fill (+3.6 % pairs/s on a B200 with two engines).
        # (private engines: model.forward() keeps its own cached one, so the two can be used side by side)
        # A pair whose size is not a multiple of 64 runs an engine of the padded size (masic_b200/padding.py): the slot
        # then holds the pair at its own size around it (x1, x2, h as submitted, the cropped x1_hat, x2_hat), and
        # everything after the codec reads those; at a multiple of 64 they are the engine's own buffers.
        first = model.engine_for(1, pad.hp, pad.wp, self.dev)          # also applies MaskedConv2d's weight masking
        self.engines = [HSICEngine(model.state_dict(), 1, pad.hp, pad.wp, self.dev, model.N, model.M, model.K,
                                   use_graph=first.use_graph) for _ in range(depth)]
        self.eng = self.engines[0]
        with torch.cuda.device(self.dev):
            self.copy_stream = torch.cuda.Stream(device=self.dev)
            self.slots = []
            for eng in self.engines:
                o = eng.out
                liks = [o["lik_y1"], o["lik_y2"], o["lik_z1"], o["lik_z2"]]
                if pad.aligned:
                    own = dict(x1=eng.x1, x2=eng.x2, h=eng.Hm, rec={"x1_hat": o["x1_hat"], "x2_hat": o["x2_hat"]})
                else:
                    img = lambda: torch.empty(1, 3, height, width, device=self.dev)   # noqa: E731
                    own = dict(x1=img(), x2=img(), h=torch.eye(3, device=self.dev).reshape(1, 3, 3),
                               rec={"x1_hat": img(), "x2_hat": img()})
                self.slots.append(dict(
                    eng=eng, stream=torch.cuda.Stream(device=self.dev), **own,
                    # criterion (8 floats) | MS-SSIM per channel of view 1 (3) and view 2 (3) | LPIPS of view 1, 2 |
                    # with enhance=True, masic_rd_metrics of the codec's (unenhanced) pair (8)
                    res_d=torch.zeros(24, device=self.dev), res_h=torch.zeros(24).pin_memory(),
                    copied=torch.cuda.Event(), done=torch.cuda.Event(), busy=False, has_result=False,
                    scratch=_ops.rd_metrics_scratch(self.dev),
                    lik_p=(C.c_void_p * 4)(*[t.data_ptr() for t in liks]),
                    lik_n=(C.c_int64 * 4)(*[t.numel() for t in liks])))
        self._ms_weights = (C.c_float * 5)(*_ops.MS_SSIM_WEIGHTS)
        self._no_lik_p, self._no_lik_n = (C.c_void_p * 4)(), (C.c_int64 * 4)()
        self._n = 0
        self.enh_out: Optional[Dict[str, torch.Tensor]] = None

    def submit(self, x1: torch.Tensor, x2: torch.Tensor, h: torch.Tensor, criterion: bool = True,
               want_recon: bool = False, msssim: bool = False, lpips: bool = False, enhance: bool = False) -> int:
        """Queue one pair.  x1 / x2: (1,3,H,W) uint8 images as they come out of the dataset's PNG files (the recommended
        host format: converted on the device exactly like torchvision's ToTensor, a quarter of the PCIe bytes, which is
        what keeps eight ranks on one host from becoming host-bound), or float32 in [0,1] as the reference's loaders
        feed them; h: (1,3,3)
        float32.  Pinned host tensors (H2D copy) or device tensors (D2D copy).  criterion=False
        skips the RateDistortionLoss reduction (forward only; `result` then just waits for the pair).  want_recon=True
        also copies the two reconstructions (what a codec is for) to pinned host memory: `reconstructions(ticket)`.
        msssim=True (with the criterion) also computes pytorch_msssim's ms_ssim(x_hat, x, data_range=1.0) of both views
        on the device (the third number of the reference's eval loop); `result` then reports it.  It needs
        min(H, W) > 160, as the package does.  lpips=True (with the criterion, after attach_lpips) also computes
        lpips.LPIPS(x_hat, x) of both views on the device (the fourth number of the eval loop).
        enhance=True (after attach_enhancement) runs full MASIC, as test3_real.py does: Independent_EN post-filters the
        decoded pair on the device, and the PSNRs, MSEs, loss, MS-SSIM, LPIPS and want_recon all refer to the enhanced
        pair; bpp still comes from the codec's likelihoods, and `result` adds the codec's own PSNR and MSE."""
        from ._lib import check
        if msssim and not criterion:
            raise ValueError("msssim=True is part of the criterion: it needs criterion=True")
        if lpips and not criterion:
            raise ValueError("lpips=True is part of the criterion: it needs criterion=True")
        s = self.slots[self._n % self.depth]
        if enhance and "cqe" not in s:
            raise MasicError("submit(enhance=True): call attach_enhancement(en) first")
        if lpips and "lpips" not in s:
            raise MasicError("submit(lpips=True): call attach_lpips(net) first")
        if msssim and "ms_scratch" not in s:
            nbytes = self.lib.masic_ms_ssim_scratch_bytes(1, 3, self.H, self.W, len(_ops.MS_SSIM_WEIGHTS))
            check(min(int(nbytes), 0), f"masic_ms_ssim_scratch_bytes ({self.H}x{self.W}: MS-SSIM needs min(H, W) > 160)")
            s["ms_scratch"] = torch.empty(nbytes, dtype=torch.uint8, device=self.dev)
        if s["busy"]:
            s["done"].synchronize()                 # the slot's previous pair has left its engine
        eng, st = s["eng"], s["stream"]
        caller = torch.cuda.current_stream(self.dev)
        self.copy_stream.wait_stream(caller)        # inputs produced on the caller's stream are complete
        as_u8 = x1.dtype == torch.uint8
        pad = self.pad
        if as_u8 and "u8" not in s:                 # 8-bit images: a quarter of the PCIe bytes, converted on the device
            s["u8"] = [torch.empty(1, 3, self.H, self.W, dtype=torch.uint8, device=self.dev) for _ in range(2)]
        with torch.cuda.stream(self.copy_stream):
            if as_u8:
                s["u8"][0].copy_(x1.reshape(1, 3, self.H, self.W), non_blocking=True)
                s["u8"][1].copy_(x2.reshape(1, 3, self.H, self.W), non_blocking=True)
            else:
                s["x1"].copy_(x1.reshape(1, 3, self.H, self.W), non_blocking=True)
                s["x2"].copy_(x2.reshape(1, 3, self.H, self.W), non_blocking=True)
            s["h"].copy_(h.reshape(1, 3, 3), non_blocking=True)
            s["copied"].record(self.copy_stream)
        with torch.cuda.stream(st):
            st.wait_event(s["copied"])
            if not pad.aligned:                     # into the padded frame; 8-bit pairs also leave the fp32 originals
                for i, (x, dst) in enumerate(((s["x1"], eng.x1), (s["x2"], eng.x2))):
                    pad.image_into(s["u8"][i] if as_u8 else x, dst, unpadded=x if as_u8 else None)
                pad.homography_into(s["h"], eng.Hm)
            elif as_u8:                             # torchvision's ToTensor: img.float().div(255), bit for bit
                for src, dst in ((s["u8"][0], eng.x1), (s["u8"][1], eng.x2)):
                    check(self.lib.masic_u8_to_unit_f32(src.data_ptr(), src.numel(), dst.data_ptr(), st.cuda_stream),
                          "masic_u8_to_unit_f32")
            o = eng.run()
            if not pad.aligned:
                for k in ("x1_hat", "x2_hat"):
                    pad.crop_into(o[k], s["rec"][k])
            codec = s["rec"]
            rec = s["cqe"].run() if enhance else codec  # the CQE graph reads the codec's x1_hat, x2_hat and h in place
            x1_, x2_ = s["x1"], s["x2"]
            if criterion:
                check(self.lib.masic_rd_metrics(s["lik_p"], s["lik_n"], rec["x1_hat"].data_ptr(), x1_.data_ptr(),
                                                rec["x2_hat"].data_ptr(), x2_.data_ptr(), 1, 3, self.H, self.W,
                                                self.lmbda, s["scratch"].data_ptr(), s["res_d"].data_ptr(),
                                                st.cuda_stream), "masic_rd_metrics")
                if enhance:                             # the codec's own MSE (no likelihoods: its bpp is the above)
                    check(self.lib.masic_rd_metrics(self._no_lik_p, self._no_lik_n, codec["x1_hat"].data_ptr(),
                                                    x1_.data_ptr(), codec["x2_hat"].data_ptr(), x2_.data_ptr(), 1, 3,
                                                    self.H, self.W, self.lmbda, s["scratch"].data_ptr(),
                                                    s["res_d"][16:].data_ptr(), st.cuda_stream), "masic_rd_metrics")
                if msssim:
                    for v, (xh, x) in enumerate(((rec["x1_hat"], x1_), (rec["x2_hat"], x2_))):
                        check(self.lib.masic_ms_ssim(xh.data_ptr(), x.data_ptr(), 1, 3, self.H, self.W, 5, 1.0, 0.01,
                                                     0.03, self._ms_weights, 1, s["ms_scratch"].data_ptr(),
                                                     s["res_d"][8 + 3 * v:].data_ptr(), st.cuda_stream), "masic_ms_ssim")
                if lpips:
                    total, _ = s["lpips_enh" if enhance else "lpips"].run(normalize=self._lpips_normalize)
                    s["res_d"][14:16].copy_(total, non_blocking=True)
                n = 24 if enhance else 16 if lpips else 14 if msssim else 8
                s["res_h"][:n].copy_(s["res_d"][:n], non_blocking=True)
            if want_recon:
                if "rec_h" not in s:
                    s["rec_h"] = [torch.empty(1, 3, self.H, self.W).pin_memory() for _ in range(2)]
                s["rec_h"][0].copy_(rec["x1_hat"], non_blocking=True)
                s["rec_h"][1].copy_(rec["x2_hat"], non_blocking=True)
            s["done"].record(st)
        s["busy"], s["has_result"], s["has_recon"], s["has_msssim"] = True, criterion, want_recon, msssim
        s["has_lpips"], s["has_enhance"] = lpips, enhance
        self.eng = eng
        self.enh_out = rec if enhance else None
        self._n += 1
        return self._n - 1

    # ---- images + grey patches in, criterion out: the homography is estimated on the device (SURVEY 8(f)#4)
    def attach_homography_net(self, net) -> None:
        """`net`: a masic_b200.udh.Net (the udh homography model, test2_real.py:42-47) on this device.  Each slot gets
        its own UDHEngine (static buffers + CUDA graph) writing h_matrix straight into the slot's codec engine."""
        from .udh import UDHEngine
        for s in self.slots:
            s["udh"] = UDHEngine(net.state_dict(), 1, self.dev, net.patch_size)

    # ---- LPIPS next to the criterion (the eval loop's fourth number)
    def attach_lpips(self, net, normalize: bool = True) -> None:
        """`net`: a masic_b200.lpips.LPIPS.  Each slot gets an LPIPSEngine of batch 4, [x1_hat, x2_hat, x1, x2], that
        reads the slot's codec buffers in place.  The stream's images are in [0, 1] (ToTensor), which lpips wants as
        forward(..., normalize=True); normalize=False reproduces a script that passes them without the flag.  Once an
        enhancement net is attached too (either order), a second engine per slot reads the enhanced pair instead."""
        self._lpips_sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
        self._lpips_normalize = bool(normalize)
        for s in self.slots:
            if s["busy"]:
                s["done"].synchronize()             # the engines replaced below may still be in use
            s["lpips"] = self._lpips_engine(s, s["rec"])
            if "cqe" in s:
                s["lpips_enh"] = self._lpips_engine(s, s["cqe"].out)

    def _lpips_engine(self, s, rec: Dict[str, torch.Tensor]):
        """An LPIPSEngine that compares the reconstructions `rec` with the slot's originals, reading both in place."""
        from .lpips import LPIPSEngine
        e = LPIPSEngine(self._lpips_sd, 2, self.H, self.W, self.dev,
                        inputs=[rec["x1_hat"], rec["x2_hat"], s["x1"], s["x2"]])
        e.prepare(self._lpips_normalize)
        return e

    # ---- full MASIC: the cross quality enhancement network after the codec (test3_real.py)
    def attach_enhancement(self, en) -> None:
        """`en`: a masic_b200.cqe.Independent_EN on this device.  Each slot gets a CQEEngine of batch 1 that reads the
        slot's codec outputs and homography in place, for submit(..., enhance=True).  The engines hold a snapshot of
        the weights taken now: call again after changing them."""
        from .cqe import CQEEngine
        sd = {k: v.detach().clone() for k, v in en.state_dict().items()}
        for s in self.slots:
            if s["busy"]:
                s["done"].synchronize()             # the engines replaced below may still be in use
            s["cqe"] = CQEEngine(sd, 1, self.H, self.W, self.dev, use_graph=en._use_graph,
                                 inputs=(s["rec"]["x1_hat"], s["rec"]["x2_hat"], s["h"]))
            if "lpips" in s:
                s["lpips_enh"] = self._lpips_engine(s, s["cqe"].out)

    def submit_patches(self, x1: torch.Tensor, x2: torch.Tensor, patch_a: torch.Tensor, patch_b: torch.Tensor,
                       corners: torch.Tensor, criterion: bool = True, want_recon: bool = False,
                       msssim: bool = False, lpips: bool = False, enhance: bool = False) -> int:
        """Like `submit`, but instead of h_matrix takes what the dataset hands over (datasets/utils.py:383-395): the two
        (1,1,128,128) normalised grey patches and their (1,4,2) corner coordinates.  The udh net, the 4-point DLT,
        the inverse and h_adjust (test2_real.py:201-211) run on the slot's stream ahead of the codec; the host never
        sees the homography."""
        s = self.slots[self._n % self.depth]
        if "udh" not in s:
            raise MasicError("submit_patches: call attach_homography_net(net) first")
        if s["busy"]:
            s["done"].synchronize()
        u = s["udh"]
        caller = torch.cuda.current_stream(self.dev)
        self.copy_stream.wait_stream(caller)
        with torch.cuda.stream(self.copy_stream):
            u.ab[:, 0:1].copy_(patch_a.reshape(1, 1, u.P, u.P), non_blocking=True)
            u.ab[:, 1:2].copy_(patch_b.reshape(1, 1, u.P, u.P), non_blocking=True)
            u.corners.copy_(corners.reshape(1, 4, 2), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        with torch.cuda.stream(s["stream"]):
            s["stream"].wait_event(ev)
            h = u.run(img_hw=(self.H, self.W), corners=u.corners)["h"]
            ev2 = torch.cuda.Event()
            ev2.record(s["stream"])
        self.copy_stream.wait_event(ev2)            # submit() copies h on the copy stream
        return self.submit(x1, x2, h, criterion=criterion, want_recon=want_recon, msssim=msssim, lpips=lpips,
                           enhance=enhance)

    def result(self, ticket: int):
        """(bpp, psnr1_db, psnr2_db, detail) of a submitted pair; blocks until its D2H copy has landed.  A pair
        submitted with msssim=True also has detail["msssim1"/"msssim2"] (mean over the 3 channels, as
        pytorch_msssim's size_average) and "msssim1_db"/"msssim2_db" = -10 log10(1 - value); one submitted with
        lpips=True has detail["lpips1"/"lpips2"].  For a pair submitted with enhance=True the PSNRs and every value
        above but the bpp are those of the enhanced pair, and detail["codec_psnr1"/"codec_psnr2"/"codec_mse1"/
        "codec_mse2"] are those of the codec's reconstructions."""
        if not (self._n - self.depth <= ticket < self._n):
            raise ValueError(f"ticket {ticket} is no longer (or not yet) in flight")
        s = self.slots[ticket % self.depth]
        s["done"].synchronize()
        if not s["has_result"]:
            return None
        r = s["res_h"].tolist()
        psnr = [10.0 * math.log10(1.0 / m) if m > 0 else float("inf") for m in r[4:6] + r[20:22]]
        detail = {"bpp_y1": r[0], "bpp_y2": r[1], "bpp_z1": r[2], "bpp_z2": r[3], "mse1": r[4], "mse2": r[5],
                  "loss": r[7]}
        if s["has_msssim"]:
            for v in (1, 2):
                m = sum(r[5 + 3 * v:8 + 3 * v]) / 3.0
                detail[f"msssim{v}"] = m
                detail[f"msssim{v}_db"] = -10.0 * math.log10(1.0 - m) if m < 1.0 else float("inf")
        if s["has_lpips"]:
            detail["lpips1"], detail["lpips2"] = r[14], r[15]
        if s["has_enhance"]:
            detail.update(codec_psnr1=psnr[2], codec_psnr2=psnr[3], codec_mse1=r[20], codec_mse2=r[21])
        return r[6], psnr[0], psnr[1], detail

    def reconstructions(self, ticket: int):
        """(x1_hat, x2_hat) of a pair submitted with want_recon=True, as pinned HOST tensors (valid until the slot is
        re-used, i.e. for the next depth-1 submissions); blocks until the D2H copies have landed."""
        if not (self._n - self.depth <= ticket < self._n):
            raise ValueError(f"ticket {ticket} is no longer (or not yet) in flight")
        s = self.slots[ticket % self.depth]
        s["done"].synchronize()
        if not s.get("has_recon"):
            raise ValueError("the pair was submitted without want_recon=True")
        return s["rec_h"][0], s["rec_h"][1]

    def outputs(self) -> Dict[str, torch.Tensor]:
        """The engine's output buffers of the last submitted pair.  For a size that is not a multiple of 64, x1_hat and
        x2_hat are the slot's cropped copies and the masks are views of the pair's window; the latents and likelihoods
        stay on the padded grid, as `HSIC.forward` returns them."""
        if self.pad.aligned:
            return self.eng.out
        s = next(s for s in self.slots if s["eng"] is self.eng)
        o = self.eng.out
        return {**o, **s["rec"], "x1_mask_R": self.pad.crop(o["x1_mask_R"]), "x1_mask_L": self.pad.crop(o["x1_mask_L"])}

    def enhanced_outputs(self) -> Dict[str, torch.Tensor]:
        """{"x1_hat", "x2_hat"} of the last submitted pair after the enhancement network, the keys of
        Independent_EN.forward: the slot's CQE output buffers (valid after `result(ticket)`, until the slot is reused).
        The last pair must have been submitted with enhance=True."""
        if self.enh_out is None:
            raise MasicError("enhanced_outputs: the last pair was submitted without enhance=True")
        return self.enh_out

    def join(self, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Make `stream` (default: the current stream) wait for every pair submitted so far (device-side, no host sync)."""
        stream = stream or torch.cuda.current_stream(self.dev)
        for s in self.slots:
            if s["busy"]:
                stream.wait_event(s["done"])


def bpp_and_psnr(out: Dict, x1: torch.Tensor, x2: torch.Tensor):
    """The criterion the reference's eval script applies to forward()'s output
    (coremasic/mywork/test2_real.py:88-114): bpp from the likelihoods, PSNR per view."""
    n, _, h, w = x1.shape
    num_pixels = n * h * w
    bpp = sum(torch.log(l).sum() / (-math.log(2) * num_pixels) for l in out["likelihoods"].values())
    mse1 = torch.mean((out["x1_hat"] - x1) ** 2)
    mse2 = torch.mean((out["x2_hat"] - x2) ** 2)
    psnr1 = 10.0 * torch.log10(1.0 / mse1)
    psnr2 = 10.0 * torch.log10(1.0 / mse2)
    return bpp, psnr1, psnr2
