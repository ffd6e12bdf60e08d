"""Cost of the exact per-voxel posterior std (``CWFAEngine.reconstruct_posterior_exact_graphed``) at the full configuration
(96 x 512 x 512, 5 steps, bf16, seeded synthetic inputs as bench.py builds them), temperature 0.7.

  * end to end, graphed, alternated within each of ``--rounds`` rounds (same process, same inputs; every timed window ends in a
    device synchronise):
      batch 1: ``reconstruct_graphed``, ``reconstruct_posterior_exact_graphed`` and ``reconstruct_posterior_graphed`` at K = 8;
      batch 8: the first two;
  * kernels: the level-0 coupling (ch 48, 512 x 512, batch 1, bf16, a row gather) as inverse ``coupling_f8`` and as
    ``coupling_f8_scale`` reading and writing the scale, and the level-0 merge (48 -> 96 channels) as ``haar1d_merge_f8`` and as
    ``haar1d_merge_std_f8`` with ``std_lo``, CUDA events over graphs of back-to-back launches, with the bytes each launch moves.

Prints the GPU name, power limit and SM clock read in the same run, then one JSON line; ``--out`` also writes the JSON."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench_posterior import gpu_info, synthetic_inputs, time_calls, time_graph


def kernel_numbers(dev):
    from cwfa_b200 import tc
    torch.manual_seed(3)
    ch, H, W, kind = 48, 512, 512, "bf16"
    P = H * W
    b8 = tc.to_c8(torch.randn((1, 64, H, W), device=dev), kind)
    w = 0.04 * torch.randn((2 * ch, 64, 3, 3), device=dev)
    bias = 0.5 * torch.randn((2 * ch,), device=dev)
    pc = tc.coupling_weights_f8(w, bias, ch, torch.arange(ch), False, kind)
    ld = torch.zeros(1, device=dev)
    ticket = torch.zeros(1, device=dev, dtype=torch.int32)
    x8 = tc.to_f8(torch.randn((1, ch, H, W), device=dev))
    s8 = tc.to_f8(torch.rand((1, ch, H, W), device=dev) + 0.5)
    rows = torch.randperm(H, generator=torch.Generator().manual_seed(4)).to(dev, torch.int32)
    kw = dict(ch=ch, perm=rows, perm_axis=2, logdet=ld, ticket=ticket)
    lo = torch.randn((1, ch, H, W), device=dev)
    std_lo = torch.rand((1, ch, H, W), device=dev)
    elems = ch * P
    cond = P * 64 * 2                                          # the bf16 trunk output read through TMA
    runs = {
        "l0_coupling_plain": (lambda: tc.coupling_f8(b8, pc, x8, inverse=True, **kw), elems * 8 + cond),
        "l0_coupling_scale": (lambda: tc.coupling_f8_scale(b8, pc, x8, s8, **kw), elems * 16 + cond),
        "l0_merge_plain": (lambda: tc.haar1d_merge_f8(lo, x8), elems * 16),                  # lo, hi in; x (2 ch) out
        "l0_merge_std": (lambda: tc.haar1d_merge_std_f8(lo, std_lo, x8, s8, 0.391), elems * 32),   # + std_lo, scale in; std out
    }
    out = {}
    for _ in range(2):                                         # alternated: two passes, the second one reported
        for name, (fn, nbytes) in runs.items():
            us = time_graph(fn, 20)
            out[f"{name}_us"] = round(us, 2)
            out[f"{name}_bytes"] = nbytes
            out[f"{name}_TBps"] = round(nbytes / us / 1e6, 3)
    out["l0_coupling_scale_over_plain"] = round(out["l0_coupling_scale_us"] / out["l0_coupling_plain_us"], 3)
    out["l0_merge_std_over_plain"] = round(out["l0_merge_std_us"] / out["l0_merge_plain_us"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--depths", type=int, default=96)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--temperature", type=float, default=0.7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_posterior_exact.py needs a CUDA device")
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    print("GPU:", info, flush=True)
    T, B = args.temperature, args.batch
    model = cwfa_b200.CWFAModel(n_depths=args.depths, volume_side_size=args.side, INN_max_down_steps=args.steps, seed=0).to(dev)
    eng = CWFAEngine(model, "bf16")
    views, mvs = synthetic_inputs(args.side, args.depths, args.steps)
    views, mvs = views.to(dev), [m.to(dev) for m in mvs]
    g = torch.Generator().manual_seed(1)
    vB = torch.cat([views] + [torch.randn(tuple(views.shape), generator=g).to(dev) for _ in range(B - 1)])
    mvB = [m.repeat(B, 1, 1, 1) for m in mvs]
    variants = {
        "b1_reconstruct": lambda: eng.reconstruct_graphed(views, mvs),
        "b1_exact": lambda: eng.reconstruct_posterior_exact_graphed(views, mvs, temperature=T),
        "b1_mc_k8": lambda: eng.reconstruct_posterior_graphed(views, mvs, 8, temperature=T),
        f"b{B}_reconstruct": lambda: eng.reconstruct_graphed(vB, mvB),
        f"b{B}_exact": lambda: eng.reconstruct_posterior_exact_graphed(vB, mvB, temperature=T),
    }
    for fn in variants.values():                               # capture and warm every graph before timing
        fn()
        fn()
    times = {name: [] for name in variants}
    for _ in range(args.rounds):
        for name, fn in variants.items():
            times[name].append(time_calls(fn, args.reps))
    res = {"gpu": info, "config": f"{args.depths}x{args.side}x{args.side} steps {args.steps} bf16, graphed, temperature {T}"}
    for name in variants:
        med = statistics.median(times[name])
        res[f"{name}_ms_per_call"] = round(med, 3)
        res[f"{name}_rounds_ms"] = [round(t, 3) for t in times[name]]
        print(f"{name:>16}: {med:.3f} ms per call  (rounds {res[f'{name}_rounds_ms']})")
    res["b1_exact_over_reconstruct"] = round(res["b1_exact_ms_per_call"] / res["b1_reconstruct_ms_per_call"], 4)
    res[f"b{B}_exact_over_reconstruct"] = round(res[f"b{B}_exact_ms_per_call"] / res[f"b{B}_reconstruct_ms_per_call"], 4)
    res["b1_mc_k8_over_exact"] = round(res["b1_mc_k8_ms_per_call"] / res["b1_exact_ms_per_call"], 4)
    kn = kernel_numbers(dev)
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
