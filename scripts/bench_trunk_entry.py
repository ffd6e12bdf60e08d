"""The first trunk block of a level's five coupling sub-networks, old pair against the composed entry launch, at 512 x 512.

Per level (LF condition of Cin = 48 / 24 / 12 / 6 channels, 5 sub-networks, bf16 and fp16):
  * pair:  the batched 1x1 input conv (Cin -> 5 x 64, ``conv_tc``) + the first batched trunk block (``resblock_tc_batched``);
  * entry: one ``resblock_tc_entry_batched`` launch that reads the condition directly.
Each is captured ``--launches`` times into one CUDA graph, inputs rotated over 8 copies (> 126 MB of L2 at Cin 48) so that no
launch reads a condition the previous one left in L2; the two forms alternate over ``--rounds`` rounds and the median per-launch
time of each is reported.  Prints the GPU name, power limit and SM clocks read in the same run, then one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"error": r.stdout + r.stderr}
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}


def graph_us(fn, launches: int) -> float:
    """Microseconds per call of ``fn(i)``, i = 0..launches-1, captured into one graph and replayed once (after a warm replay)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(3):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(launches):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--launches", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--kinds", default="bf16,fp16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_trunk_entry.py measures on the GPU; no CUDA device found")
    import cwfa_b200  # noqa: F401
    from cwfa_b200 import tc
    from oracle.weights import seeded_randn

    info = gpu_info()
    print(f"GPU: {info.get('name')}  power limit {info.get('power.limit')}  SM clock {info.get('clocks.sm')} "
          f"(max {info.get('clocks.max.sm')})", flush=True)
    dev, S, nsets, nrot = "cuda:0", args.side, 5, 8
    rows = []
    for kind in args.kinds.split(","):
        for cin in (48, 24, 12, 6):
            lfs = [tc.to_c8(seeded_randn((1, cin, S, S), 1 + i).to(dev), kind) for i in range(nrot)]
            subs = []
            for k in range(nsets):
                win = seeded_randn((64, cin, 1, 1), 10 * k + 2, (1.0 / cin) ** 0.5).to(dev)
                bin_ = seeded_randn((64,), 10 * k + 3, 0.1).to(dev)
                w3 = seeded_randn((64, 64, 3, 3), 10 * k + 4, (1.0 / 576) ** 0.5).to(dev)
                b3 = seeded_randn((64,), 10 * k + 5, 0.1).to(dev)
                p1 = tc.PackedConv(seeded_randn((64, 64, 1, 1), 10 * k + 6, 0.125).to(dev), seeded_randn((64,), 10 * k + 7, 0.1).to(dev),
                                   kind, bn=64)
                subs.append((win, bin_, w3, b3, p1))
            batched_in = tc.PackedConv(torch.cat([s[0] for s in subs]), torch.cat([s[1] for s in subs]), kind, bn=64)
            sets = [(tc.PackedConv(s[2], s[3], kind, bn=64), s[4]) for s in subs]
            entries = [tc.PackedEntry(s[0], s[1], s[2], s[3], s[4], kind) for s in subs]

            def pair(i):
                tc.resblock_tc_batched(tc.conv_tc(lfs[i % nrot], batched_in), sets)

            def entry(i):
                tc.resblock_tc_entry_batched(lfs[i % nrot], entries)

            t_pair, t_entry = [], []
            for _ in range(args.rounds):
                t_pair.append(graph_us(pair, args.launches))
                t_entry.append(graph_us(entry, args.launches))
            mp, me = statistics.median(t_pair), statistics.median(t_entry)
            row = dict(kind=kind, cin=cin, pair_us=round(mp, 2), entry_us=round(me, 2), ratio=round(me / mp, 3),
                       pair_spread_us=round(max(t_pair) - min(t_pair), 2), entry_spread_us=round(max(t_entry) - min(t_entry), 2))
            rows.append(row)
            print(f"{kind} Cin {cin:2d}: 1x1 conv + block {mp:7.1f} us   entry {me:7.1f} us   ratio {me / mp:.3f}   "
                  f"(spread {row['pair_spread_us']} / {row['entry_spread_us']} us)", flush=True)
            del lfs
            torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=info, side=S, sets=nsets, rows=rows)))


if __name__ == "__main__":
    main()
