"""Batched coding of stereo pairs: HSIC.compress_batch / decompress_batch pairs/s against the per-pair file API.

    python tools/codec_batch_bench.py [--batches 1,2,4,8,16] [--rounds 3] [--roundtrip-json this.json parent.json ...]
                                      [--out profiles/r3_codec_batch_n1.json]

Workloads (BASELINE.json configs[3] and configs[2] geometry), HSIC seed 0 with g_a_conv4 x 8 so that the latents are
not all zero (at random init every y symbol is 0), inputs uniform noise (the largest payloads):
  full   16 distinct pairs of 1216x2176; batch B codes pairs 0..B-1
  small  64 pairs of 512x512, coded in 64 / B calls of B pairs
Configurations (one per B and workload) are alternated round by round.  Each configuration's first call of a round
builds its engine (`engine_for` keeps one), so every round times the second and third calls: compress_batch and
decompress_batch, host wall clock around the call with a device synchronise on either side.  Every batch result is
checked byte for byte (payloads) and bit for bit (latents, reconstructions) against B = 1 of the same path.
After the rounds, one decompress_batch call per B of the full workload runs under torch.profiler (CUDA activity only):
the summed device time of its kernels and copies over the 2 x 361 waves is the GPU time per wave, next to the host
wall time per wave of the timed calls.
`--roundtrip-json` takes the JSON lines `bench.py --blocks codec_roundtrip` printed on this tree and on the parent
tree (label=path) and records their per-pair compress / decompress times beside these numbers."""
import argparse
import gc
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from masic_b200.bitstream import wave_schedule  # noqa: E402
from masic_b200.hsic import HSIC  # noqa: E402
from oracle.hsic import synthetic_homography  # noqa: E402
from tools.lpips_bench import gpu_info  # noqa: E402

KEYS = ("x1_hat", "x2_hat", "y1_hat", "y2_hat", "z1_hat", "z2_hat")


def sync_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def code_all(net, x1, x2, Hm, B):
    """Compress then decompress all pairs in calls of B; returns (compress s, decompress s, items, decoded)."""
    n = x1.shape[0]
    items, outs, tc, td = [], [], 0.0, 0.0
    for i in range(0, n, B):
        it, t = sync_time(lambda: net.compress_batch(x1[i:i + B], x2[i:i + B], Hm[i:i + B]))
        tc += t
        items += it
    for i in range(0, n, B):
        o, t = sync_time(lambda: net.decompress_batch([(d["header"], d["payload"]) for d in items[i:i + B]],
                                                      Hm[i:i + B]))
        td += t
        outs.append(o)
    return tc, td, items, {k: torch.cat([o[k] for o in outs]) for k in KEYS}


def device_ms(fn):
    """Summed device time (ms) of the kernels and copies fn issues, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(getattr(e, "self_device_time_total", 0.0) for e in prof.key_averages()) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,2,4,8,16")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--roundtrip-json", nargs="*", default=[], help="label=path of a bench.py codec_roundtrip line")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_codec_batch_n1.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("codec_batch_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    batches = [int(b) for b in a.batches.split(",")]
    info = gpu_info(0)
    torch.manual_seed(0)
    net = HSIC().eval()
    with torch.no_grad():
        net.encoder1.g_a_conv4.weight.mul_(8.0)
        net.encoder2.g_a_conv4.weight.mul_(8.0)
    net = net.to(dev)
    net.update(force=True)
    g = torch.Generator().manual_seed(7)
    work = {}
    for name, n, h, w in (("full", max(batches), 1216, 2176), ("small", 64, 512, 512)):
        x1 = torch.rand(n, 3, h, w, generator=g).to(dev)
        x2 = torch.rand(n, 3, h, w, generator=g).to(dev)
        work[name] = (x1, x2, synthetic_homography(n, seed=3).to(dev))
    res = {name: {B: {"compress_s": [], "decompress_s": [], "max_memory_allocated_GB": 0.0} for B in batches}
           for name in work}
    exact = True
    with torch.no_grad():
        # B = 1 of the same path over every pair of a workload: the reference each batch result must equal
        ref = {name: code_all(net, *work[name], 1)[2:] for name in work}
        for rnd in range(a.rounds):
            for name, (x1, x2, Hm) in work.items():
                for B in batches:
                    n = B if name == "full" else x1.shape[0]
                    args = (net, x1[:n], x2[:n], Hm[:n], B)
                    code_all(*args)                                  # builds the batch-B engine and its wave models
                    gc.collect()             # an engine and its cached wave models form a cycle: free the replaced ones
                    torch.cuda.reset_peak_memory_stats(dev)
                    for _ in range(2):
                        tc, td, items, out = code_all(*args)
                        res[name][B]["compress_s"].append(tc)
                        res[name][B]["decompress_s"].append(td)
                    r = res[name][B]
                    r["max_memory_allocated_GB"] = max(r["max_memory_allocated_GB"], torch.cuda.max_memory_allocated(dev) / 1e9)
                    r["pairs"] = n
                    ritems, rout = ref[name]
                    exact &= all(it["header"] == q["header"] and it["payload"] == q["payload"] for it, q in zip(items, ritems))
                    exact &= all(torch.equal(out[k], rout[k][:n]) for k in KEYS)
                    print(rnd, name, B, f"compress {n / tc:.2f} pairs/s, decompress {n / td:.2f} pairs/s", flush=True)
    waves = 2 * len(wave_schedule(1216 // 16, 2176 // 16))
    per_wave = {}
    with torch.no_grad():
        x1, x2, Hm = work["full"]
        for B in batches:
            items = net.compress_batch(x1[:B], x2[:B], Hm[:B])
            pairs = [(d["header"], d["payload"]) for d in items]
            net.decompress_batch(pairs, Hm[:B])
            try:
                gpu = device_ms(lambda: net.decompress_batch(pairs, Hm[:B]))
            except Exception as e:                          # report, do not guess
                per_wave[str(B)] = {"error": repr(e)}
                continue
            host = min(res["full"][B]["decompress_s"]) * 1e3
            per_wave[str(B)] = {"decompress_ms": host, "device_busy_ms": gpu, "waves": waves,
                                "host_ms_per_wave": host / waves, "device_ms_per_wave": gpu / waves}
            print("per wave", B, per_wave[str(B)], flush=True)
    summary = {}
    for name in work:
        summary[name] = {}
        for B in batches:
            r = res[name][B]
            n = r["pairs"]
            summary[name][str(B)] = {
                "pairs": n,
                "compress_pairs_per_s": [n / t for t in r["compress_s"]],
                "decompress_pairs_per_s": [n / t for t in r["decompress_s"]],
                "compress_vs_B1": max(n / t for t in r["compress_s"]) / max(
                    res[name][1]["pairs"] / t for t in res[name][1]["compress_s"]) if 1 in res[name] else None,
                "decompress_vs_B1": max(n / t for t in r["decompress_s"]) / max(
                    res[name][1]["pairs"] / t for t in res[name][1]["decompress_s"]) if 1 in res[name] else None,
                "max_memory_allocated_GB": r["max_memory_allocated_GB"],
            }
    roundtrip = {}
    for spec in a.roundtrip_json:
        label, path = spec.split("=", 1)
        line = json.loads([ln for ln in Path(path).read_text().splitlines() if ln.startswith("{")][-1])
        roundtrip[label] = line["codec_roundtrip"]
    if "parent" in roundtrip and "full" in summary:
        par = roundtrip["parent"]
        for B, s in summary["full"].items():
            s["compress_vs_parent_per_pair"] = max(s["compress_pairs_per_s"]) * par["compress_ms"] / 1e3
            s["decompress_vs_parent_per_pair"] = max(s["decompress_pairs_per_s"]) * par["decompress_ms"] / 1e3
    doc = {"tool": "tools/codec_batch_bench.py", **info, "rounds": a.rounds,
           "workloads": {"full": "1216x2176 noise pairs, batch B codes B pairs", "small": "64 512x512 noise pairs in 64/B calls"},
           "batch_equals_B1_bit_exact": bool(exact), "results": summary,
           "decompress_per_wave_full": per_wave, "per_pair_file_api": roundtrip}
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(doc, indent=1) + "\n")
    print(json.dumps({"gpu": info, "exact": exact}))


if __name__ == "__main__":
    main()
