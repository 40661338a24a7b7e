"""Pairs of any size (masic_b200/padding.py) on one GPU: what the pad and crop around the 64-multiple engine cost.

    python tools/any_size_bench.py [--pairs 6] [--stream-pairs 96] [--rounds 3] [--out profiles/r3_any_size_n1.json]

  a  PairStream pairs/s at 375x1242 (KITTI; padded to 384x1280) against 384x1280, pinned 8-bit host pairs rotating over
     `--pairs` distinct pairs, depth 3, criterion on, the two configurations alternated round by round.  Host wall clock
     over a round, every result read back.
  b  masic_pad_image per pair: two launches (8-bit source -> padded fp32 frame + the fp32 original), CUDA events over
     `--iters` pairs rotating over the buffers of 10 pairs (258 MB, more than the L2), and the bandwidth against the
     algorithmic bytes n*c*(h*w*1 + Hp*Wp*4 + h*w*4) per launch.
  c  compress_batch / decompress_batch at B = 8 at 375x1242 (HSIC seed 0 with g_a_conv4 x 8), seconds per call after
     one warm-up call, median over rounds.
Random-init weights: the kernels' cost does not depend on the weights' values."""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from masic_b200.hsic import HSIC  # noqa: E402
from masic_b200.padding import padding_for  # noqa: E402
from oracle.hsic import synthetic_homography  # noqa: E402
from tools.lpips_bench import gpu_info, timed  # noqa: E402


def stream_rate(ps, pairs, n):
    t0 = time.perf_counter()
    tickets = []
    for i in range(n):
        x1, x2, h = pairs[i % len(pairs)]
        tickets.append(ps.submit(x1, x2, h))
        if i >= ps.depth - 1:
            ps.result(tickets[i - ps.depth + 1])
    for t in tickets[-(ps.depth - 1):]:
        ps.result(t)
    return n / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=6)
    ap.add_argument("--stream-pairs", type=int, default=96)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_any_size_n1.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("any_size_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    torch.manual_seed(0)
    net = HSIC().eval()
    with torch.no_grad():
        net.encoder1.g_a_conv4.weight.mul_(8.0)
        net.encoder2.g_a_conv4.weight.mul_(8.0)
    net = net.to(dev)
    net.update(force=True)
    g = torch.Generator().manual_seed(7)
    sizes = {"375x1242": (375, 1242), "384x1280": (384, 1280)}
    host = {k: [tuple(t.pin_memory() for t in (torch.randint(0, 256, (1, 3, h, w), generator=g, dtype=torch.uint8),
                                                 torch.randint(0, 256, (1, 3, h, w), generator=g, dtype=torch.uint8),
                                                 synthetic_homography(1, seed=i)))
                for i in range(a.pairs)] for k, (h, w) in sizes.items()}
    doc = {**info, "torch": torch.__version__}
    with torch.no_grad():
        # a: the pair stream, alternated
        streams = {k: net.pair_stream(h, w, dev, depth=3, lmbda=0.001) for k, (h, w) in sizes.items()}
        for k, ps in streams.items():
            stream_rate(ps, host[k], 2 * ps.depth)                 # graph capture, warm-up
        rates = {k: [] for k in sizes}
        for _ in range(a.rounds):
            for k, ps in streams.items():
                rates[k].append(stream_rate(ps, host[k], a.stream_pairs))
        doc["pair_stream_pairs_per_s"] = rates
        med = {k: statistics.median(v) for k, v in rates.items()}
        doc["pair_stream_ratio_375x1242_over_384x1280"] = med["375x1242"] / med["384x1280"]
        doc["pixels_ratio_384x1280_over_375x1242"] = 384 * 1280 / (375 * 1242)
        del streams
        torch.cuda.empty_cache()

        # b: the pad kernel, rotating over buffers of 10 pairs (258 MB > the 126 MB L2)
        pad = padding_for(375, 1242)
        bufs = [([torch.randint(0, 256, (1, 3, pad.h, pad.w), generator=g, dtype=torch.uint8).to(dev) for _ in range(2)],
                 [torch.empty(1, 3, pad.hp, pad.wp, device=dev) for _ in range(2)],
                 [torch.empty(1, 3, pad.h, pad.w, device=dev) for _ in range(2)]) for _ in range(10)]

        def one_pair(i):
            src, dst, orig = bufs[i % len(bufs)]
            for v in range(2):
                pad.image_into(src[v], dst[v], unpadded=orig[v])
        ms = timed(one_pair, a.iters)
        nbytes = 2 * 3 * (pad.h * pad.w * (1 + 4) + pad.hp * pad.wp * 4)
        doc["pad_image_per_pair"] = {"ms": ms, "bytes": nbytes, "GB_per_s": nbytes / (ms * 1e-3) / 1e9,
                                     "launches": 2, "working_set": "10 pairs of buffers rotated, 258 MB (> L2)"}
        del bufs

        # c: batched coding at B = 8
        x1 = torch.rand(8, 3, 375, 1242, generator=g).to(dev)
        x2 = torch.rand(8, 3, 375, 1242, generator=g).to(dev)
        Hm = synthetic_homography(8, seed=3).to(dev)
        items = net.compress_batch(x1, x2, Hm)
        net.decompress_batch([(it["header"], it["payload"]) for it in items], Hm)
        tc, td = [], []
        for _ in range(a.rounds):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            items = net.compress_batch(x1, x2, Hm)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            net.decompress_batch([(it["header"], it["payload"]) for it in items], Hm)
            torch.cuda.synchronize()
            tc.append(t1 - t0)
            td.append(time.perf_counter() - t1)
        doc["codec_batch_375x1242_B8"] = {"compress_s": tc, "decompress_s": td,
                                         "compress_pairs_per_s": 8 / statistics.median(tc),
                                         "decompress_pairs_per_s": 8 / statistics.median(td),
                                         "bpp_real": [it["bpp_real"] for it in items]}
    print(json.dumps(doc, indent=1))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    main()
