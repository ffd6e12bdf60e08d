"""Cost of the per-voxel NLL maps of ``CWFAEngine.forward_nll_graphed(nll_map=True)`` at the full configuration (96 x 512 x 512,
5 steps, bf16, batch 8, seeded synthetic inputs as bench.py builds them).

  * end to end: ``forward_nll_graphed`` without and with maps, alternated within each of ``--rounds`` rounds (same process,
    same inputs); every timed window ends in a device synchronise; frames/s = batch / time per call;
  * kernel: the level-0 coupling (ch 48, 512 x 512, batch 8, bf16) as ``coupling_f8`` and as ``coupling_f8_map`` in its
    first-block mode (map written) and its middle-block mode (map read and written), CUDA events over graphs of back-to-back
    launches, with the bytes each launch must move and the rate they imply.

Prints the GPU name, power limit and SM clock read in the same run, then one JSON line; ``--out`` also writes the JSON."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench_posterior import gpu_info, time_calls, time_graph


def synthetic_batch(B, side, depths, steps, seed=0):
    """Volumes and views N(0, 1), the mean-volume pyramid 0.1 N(0, 1) repeated over the batch (bench.py's forward inputs)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    vol = torch.randn((B, depths, side, side), generator=g)
    views = torch.randn((B, 29, side, side), generator=g)
    mvs = [0.1 * torch.randn((1, depths // 2 ** (n + 1), side, side), generator=g).repeat(B, 1, 1, 1) for n in range(steps - 1)]
    return vol, views, mvs


def kernel_numbers(B, dev):
    from cwfa_b200 import tc
    torch.manual_seed(3)
    ch, H, W, kind = 48, 512, 512, "bf16"
    b8 = tc.to_c8(torch.randn((B, 64, H, W), device=dev), kind)
    w = 0.04 * torch.randn((2 * ch, 64, 3, 3), device=dev)
    bias = 0.5 * torch.randn((2 * ch,), device=dev)
    pc = tc.coupling_weights_f8(w, bias, ch, torch.arange(ch), False, kind)
    ld, sq = torch.zeros(B, device=dev), torch.zeros(B, device=dev)
    ticket = torch.zeros(1, device=dev, dtype=torch.int32)
    x8 = tc.to_f8(torch.randn((B, ch, H, W), device=dev))
    m8 = torch.zeros_like(x8)
    g = torch.Generator().manual_seed(4)
    rows = torch.randperm(H, generator=g).to(dev, torch.int32)
    cols = torch.randperm(W, generator=g).to(dev, torch.int32)
    elems = B * ch * H * W
    cond = B * H * W * 64 * 2                                  # the bf16 trunk output read through TMA
    # every variant gathers x through the same row permutation; the map tables permute rows and columns, as a level's later
    # blocks do
    kw = dict(ch=ch, perm=rows, perm_axis=2, logdet=ld, sumsq=sq, ticket=ticket)
    runs = {
        "plain": (lambda: tc.coupling_f8(b8, pc, x8, inverse=False, **kw), 8),
        "map_first": (lambda: tc.coupling_f8_map(b8, pc, x8, m8, map_mode=tc.NLL_MAP_FIRST, row_src=rows, col_src=cols, **kw), 12),
        "map_middle": (lambda: tc.coupling_f8_map(b8, pc, x8, m8, map_mode=0, row_src=rows, col_src=cols, **kw), 16),
    }
    out = {}
    for _ in range(2):                                         # alternated: two passes, the second one reported
        for name, (fn, bpe) in runs.items():
            us = time_graph(fn, 20)
            nbytes = elems * bpe + cond
            out[f"l0_coupling_{name}_us"] = round(us, 2)
            out[f"l0_coupling_{name}_bytes"] = nbytes
            out[f"l0_coupling_{name}_TBps"] = round(nbytes / us / 1e6, 3)
    out["l0_coupling_middle_over_plain"] = round(out["l0_coupling_map_middle_us"] / out["l0_coupling_plain_us"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--depths", type=int, default=96)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_nll_map.py needs a CUDA device")
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    print("GPU:", info, flush=True)
    B = args.batch
    model = cwfa_b200.CWFAModel(n_depths=args.depths, volume_side_size=args.side, INN_max_down_steps=args.steps, seed=0).to(dev)
    eng = CWFAEngine(model, "bf16")
    vol, views, mvs = synthetic_batch(B, args.side, args.depths, args.steps)
    vol, views, mvs = vol.to(dev), views.to(dev), [m.to(dev) for m in mvs]
    variants = {"plain": lambda: eng.forward_nll_graphed(vol, views, mvs),
                "nll_map": lambda: eng.forward_nll_graphed(vol, views, mvs, nll_map=True)}
    for fn in variants.values():                               # capture and warm both graphs before timing
        fn()
        fn()
    times = {name: [] for name in variants}
    for _ in range(args.rounds):
        for name, fn in variants.items():
            times[name].append(time_calls(fn, args.reps))
    res = {"gpu": info, "config": f"{args.depths}x{args.side}x{args.side} steps {args.steps} bf16 batch {B}, graphed"}
    for name in variants:
        med = statistics.median(times[name])
        res[f"{name}_ms_per_call"] = round(med, 3)
        res[f"{name}_frames_per_s"] = round(B * 1e3 / med, 1)
        res[f"{name}_rounds_ms"] = [round(t, 3) for t in times[name]]
        print(f"{name:>8}: {med:.3f} ms per batch of {B} = {B * 1e3 / med:.1f} frames/s  (rounds {res[f'{name}_rounds_ms']})")
    res["nll_map_over_plain"] = round(res["nll_map_ms_per_call"] / res["plain_ms_per_call"], 4)
    print(f"maps cost {100 * (res['nll_map_over_plain'] - 1):.1f} % of the map-free call")
    kn = kernel_numbers(B, dev)
    res.update(kn)
    for k, v in kn.items():
        print(f"  {k}: {v}")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
