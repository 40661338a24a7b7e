"""Full MASIC evaluation (test3_real.py: codec, then the cross quality enhancement network, then bpp, PSNR, MS-SSIM and
LPIPS of the enhanced pair) at 1216x2176 on one GPU, through PairStream and through today's one-call-at-a-time path.

    python tools/masic_stream_bench.py [--pairs 6] [--stream-pairs 48] [--rounds 3] [--out profiles/r3_masic_stream_n1.json]

Configurations, alternated round by round on pinned 8-bit host pairs (rotating over `--pairs` distinct pairs, 15.9 MB
each, so the inputs alone exceed the 126 MB L2; a CQE pass streams several GB of activations):
  a  PairStream.submit()                                        the codec stream alone
  b  PairStream.submit(enhance=True)                            codec + CQE, criterion of the enhanced pair
  c  PairStream.submit(enhance=True, msssim=True, lpips=True)   the full test3 row
  d  HSIC.forward -> Independent_EN.forward -> ops.ms_ssim -> LPIPS -> .item(), one pair at a time
Pairs/s are host wall-clock over a round, results read back for every pair.  One codec and one CQE graph replay are
also timed with CUDA events, rotating over the stream's slots (e).  Random-init weights (HSIC seed 0, Independent_EN
seed 3, LPIPS oracle seed 0): the kernels' cost does not depend on the weights' values."""
import argparse
import json
import math
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from masic_b200 import ops  # noqa: E402
from masic_b200.cqe import Independent_EN  # noqa: E402
from masic_b200.hsic import HSIC, bpp_and_psnr  # noqa: E402
from masic_b200.lpips import LPIPS  # noqa: E402
from oracle import hsic as OH  # noqa: E402
from oracle import lpips as OL  # noqa: E402
from tools.lpips_bench import gpu_info, timed  # noqa: E402

GB = 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=6, help="distinct host pairs the rounds rotate over")
    ap.add_argument("--stream-pairs", type=int, default=48, help="pairs per round")
    ap.add_argument("--rounds", type=int, default=3, help="rounds per configuration (alternating)")
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--iters", type=int, default=30, help="graph replays per CUDA-event timing")
    ap.add_argument("--height", type=int, default=1216)
    ap.add_argument("--width", type=int, default=2176)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_masic_stream_n1.json"))
    a = ap.parse_args()
    if a.pairs < 6:
        ap.error("--pairs must be >= 6 (the rotation has to exceed the L2)")
    if not torch.cuda.is_available():
        raise SystemExit("masic_stream_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    H, W = a.height, a.width
    info = gpu_info(0)
    torch.manual_seed(0)
    codec = HSIC().eval().to(dev)
    torch.manual_seed(3)
    en = Independent_EN().eval().to(dev)
    lp = LPIPS(pretrained=False, pnet_rand=True, verbose=False)
    lp.load_state_dict(OL.random_state_dict(0))
    lp = lp.to(dev)
    gh = torch.Generator().manual_seed(1)
    u = [(torch.randint(0, 256, (1, 3, H, W), generator=gh, dtype=torch.uint8).pin_memory(),
          torch.randint(0, 256, (1, 3, H, W), generator=gh, dtype=torch.uint8).pin_memory()) for _ in range(a.pairs)]
    hs = [h.reshape(1, 3, 3).contiguous().pin_memory() for h in OH.synthetic_homography(a.pairs, seed=1)]

    # ---- engines, built in configuration order; max_memory_allocated after each configuration's first round
    mem = {}
    ps = codec.pair_stream(H, W, dev, depth=a.depth)

    def stream_round(kw, n):
        t0 = time.perf_counter()
        tickets, last = [], None
        for i in range(n):
            j = i % a.pairs
            tickets.append(ps.submit(u[j][0], u[j][1], hs[j], **kw))
            if i >= ps.depth - 1:
                last = ps.result(tickets[i - ps.depth + 1])
        for t in tickets[max(0, n - ps.depth + 1):]:
            last = ps.result(t)
        return n / (time.perf_counter() - t0), last

    def today(n):
        """test3_real.py's loop on the public modules: device copy, forward, forward, metrics, .item() per number."""
        t0 = time.perf_counter()
        row = None
        with torch.no_grad():
            for i in range(n):
                j = i % a.pairs
                x1 = u[j][0].to(dev, non_blocking=True).float().div(255)
                x2 = u[j][1].to(dev, non_blocking=True).float().div(255)
                hm = hs[j].to(dev, non_blocking=True)
                out = codec(x1, x2, hm)
                enh = en(out["x1_hat"], out["x2_hat"], hm)
                bpp, p1, p2 = bpp_and_psnr({"likelihoods": out["likelihoods"], **enh}, x1, x2)
                row = [bpp.item(), p1.item(), p2.item(),
                       ops.ms_ssim(enh["x1_hat"], x1, data_range=1.0).item(),
                       ops.ms_ssim(enh["x2_hat"], x2, data_range=1.0).item(),
                       lp(enh["x1_hat"], x1, normalize=True).item(), lp(enh["x2_hat"], x2, normalize=True).item()]
        return n / (time.perf_counter() - t0), row

    configs = {"a_codec_stream": lambda n: stream_round({}, n),
               "b_enhance": lambda n: stream_round({"enhance": True}, n),
               "c_enhance_msssim_lpips": lambda n: stream_round({"enhance": True, "msssim": True, "lpips": True}, n),
               "d_today_one_pair_at_a_time": today}
    for name, fn in configs.items():
        if name == "b_enhance":
            ps.attach_enhancement(en)
        elif name == "c_enhance_msssim_lpips":
            ps.attach_lpips(lp, normalize=True)
        torch.cuda.reset_peak_memory_stats(dev)
        fn(2 * a.pairs)                                # warm-up: graph captures, module loads
        torch.cuda.synchronize()
        mem[name] = torch.cuda.max_memory_allocated(dev) / GB

    # ---- (e) one graph replay each, CUDA events, rotating over the slots
    slots = ps.slots
    t_codec = timed(lambda i: slots[i % len(slots)]["eng"].graph.replay(), a.iters)
    t_cqe = timed(lambda i: slots[i % len(slots)]["cqe"].graph.replay(), a.iters)

    # ---- pairs/s, configurations alternating round by round
    rates = {k: [] for k in configs}
    rows = {}
    for _ in range(a.rounds):
        for name, fn in configs.items():
            r, rows[name] = fn(a.stream_pairs)
            rates[name].append(r)
    med = {k: sorted(v)[len(v) // 2] for k, v in rates.items()}
    bar = 0.95 * 1000.0 / (t_codec + t_cqe)

    # the full row of the last pair, stream (c) against today's path (d): the same pair (rounds are multiples of
    # --pairs apart), so they must agree up to the order of the final mean over 3 channels
    c, d = rows["c_enhance_msssim_lpips"], rows["d_today_one_pair_at_a_time"]
    c_row = [c[0], c[1], c[2], c[3]["msssim1"], c[3]["msssim2"], c[3]["lpips1"], c[3]["lpips2"]]
    same_pair = a.stream_pairs % a.pairs == 0
    diff = [abs(x - y) for x, y in zip(c_row, d)]

    res = {
        "metric": "full MASIC (codec + CQE + bpp/PSNR/MS-SSIM/LPIPS of the enhanced pair) pairs/s, 1216x2176",
        "height": H, "width": W, **info, "device_count": torch.cuda.device_count(),
        "depth": a.depth, "distinct_host_pairs": a.pairs, "pairs_per_round": a.stream_pairs, "rounds": a.rounds,
        "pairs_per_s": rates, "pairs_per_s_median": med,
        "codec_graph_ms": t_codec, "cqe_graph_ms": t_cqe, "graph_replays_timed": a.iters,
        "bar_b_pairs_per_s": bar, "b_over_bar": med["b_enhance"] / bar,
        "b_over_graph_bound": med["b_enhance"] * (t_codec + t_cqe) / 1000.0,
        "c_over_d": med["c_enhance_msssim_lpips"] / med["d_today_one_pair_at_a_time"],
        "max_memory_allocated_gb": mem,
        "max_memory_note": "cumulative, in the order a, b, c, d: each value is the peak during that configuration's "
                           "first round with every engine of the earlier configurations still allocated (a includes "
                           "the codec engine PairStream's constructor caches on the model)",
        "last_pair_stream_vs_today": {"same_pair": same_pair, "stream_c": c_row, "today_d": d,
                                      "max_abs_diff": max(diff) if all(map(math.isfinite, diff)) else None},
        "multi_gpu": "not measured",
        "setup": f"HSIC seed 0, Independent_EN seed 3, LPIPS(alex) oracle weights seed 0 with normalize=True; PairStream "
                 f"depth {a.depth}; pinned uint8 host pairs and float32 homographies; criterion read back every pair; "
                 f"(e) CUDA events over {a.iters} replays rotating over the {a.depth} slots after a device-side sleep",
    }
    print(json.dumps(res))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
