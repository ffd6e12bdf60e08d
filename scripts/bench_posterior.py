"""Posterior statistics over K latent samples at the full configuration (96 x 512 x 512, 5 steps, bf16, seeded synthetic inputs
as bench.py builds them, temperature 0.7).

For each K in --ks, alternated within each round (same process, same inputs):
  * posterior: ``reconstruct_posterior_graphed(n_samples=K)`` -> (mean, std);
  * multi:     ``reconstruct_graphed(n_samples=K)``, the existing mean-only path;
  * singles:   K single-sample ``reconstruct_graphed`` replays into a (K, D, H, W) buffer, then torch mean / std.
Every call samples its latents outside the graph (trunc_normal_) and ends in a device synchronise; times are CUDA events.

Kernels (CUDA events over graphs of back-to-back launches): the level-0 coupling (ch 48, 512 x 512, bf16) as the K-sample
kernel against the single-sample kernel, and the level-0 merge with statistics against the bytes it must move.
Prints the GPU name, power limit and SM clock read in the same run, then one JSON line; ``--out`` also writes the JSON."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

HBM_TBPS = 7.7


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"error": r.stdout + r.stderr}
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}


def synthetic_inputs(side, depths, steps, seed=0):
    """bench.py's synthetic_inputs: views N(0,1) (1,29,S,S); mean-volume pyramid 0.1*N(0,1)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    views = torch.randn((1, 29, side, side), generator=g)
    mvs = [0.1 * torch.randn((1, depths // 2 ** (n + 1), side, side), generator=g) for n in range(steps - 1)]
    mvs.append(0.1 * torch.randn((1, depths // 2 ** (steps - 1), side, side), generator=g))
    return views, mvs


def time_calls(fn, reps: int) -> float:
    """Milliseconds per call of ``fn`` (reps calls between two events, synchronised)."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def time_graph(fn, launches: int, reps: int = 5) -> float:
    """Microseconds per launch of ``fn()`` captured ``launches`` times into one graph (median over ``reps`` replays)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(launches):
            fn()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / launches)
    return statistics.median(ts)


def kernel_numbers(ks, dev):
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
    out = {}
    x1 = tc.to_f8(torch.randn((1, ch, H, W), device=dev))
    single = time_graph(lambda: tc.coupling_f8(b8, pc, x1, ch=ch, inverse=True, logdet=ld, ticket=ticket), 20)
    out["coupling_single_us"] = round(single, 2)
    for K in ks:
        xk = tc.to_f8(torch.randn((K, ch, H, W), device=dev))
        tk = time_graph(lambda: tc.coupling_f8_samples(b8, pc, xk, K, ch=ch, logdet=ld, ticket=ticket), 20)
        moved = 2 * K * ch * P * 4                                 # x in, y out (bytes of the samples; the C8 input is 32 MB)
        out[f"coupling_K{K}_us"] = round(tk, 2)
        out[f"coupling_K{K}_per_extra_sample_us"] = round((tk - single) / (K - 1), 2)
        out[f"coupling_K{K}_xy_TBps"] = round(moved / tk / 1e6, 3)
        # level-0 merge with statistics: lo (K rows, 48 ch) + hi (K rows F8, 48 ch) in, mean + std (96 ch) out
        lo = torch.randn((K, ch, H, W), device=dev)
        ts = time_graph(lambda: tc.haar1d_merge_stats(lo, xk), 20)
        nbytes = K * 2 * ch * P * 4 + 2 * 2 * ch * P * 4
        out[f"stats_K{K}_us"] = round(ts, 2)
        out[f"stats_K{K}_bytes"] = nbytes
        out[f"stats_K{K}_TBps"] = round(nbytes / ts / 1e6, 3)
        out[f"stats_K{K}_share_of_7.7TBps"] = round(nbytes / ts / 1e6 / HBM_TBPS, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,4,8,16")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--temperature", type=float, default=0.7)
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--depths", type=int, default=96)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_posterior.py needs a CUDA device")
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    print("GPU:", info, flush=True)
    ks = [int(k) for k in args.ks.split(",")]
    T = args.temperature
    model = cwfa_b200.CWFAModel(n_depths=args.depths, volume_side_size=args.side, INN_max_down_steps=args.steps, seed=0).to(dev)
    eng = CWFAEngine(model, "bf16")
    views, mvs = synthetic_inputs(args.side, args.depths, args.steps)
    views, mvs = views.to(dev), [m.to(dev) for m in mvs]
    bufs = {K: torch.empty((K, args.depths, args.side, args.side), device=dev) for K in ks}

    def singles(K):
        for k in range(K):
            bufs[K][k].copy_(eng.reconstruct_graphed(views, mvs, temperature=T)[0])
        return torch.std_mean(bufs[K], dim=0, keepdim=True)

    variants = {
        "posterior": lambda K: eng.reconstruct_posterior_graphed(views, mvs, K, temperature=T),
        "multi": lambda K: eng.reconstruct_graphed(views, mvs, n_samples=K, temperature=T),
        "singles": singles,
    }
    for K in ks:                                            # capture / warm every graph before timing
        for fn in variants.values():
            fn(K)
            fn(K)
    eng.reconstruct_graphed(views, mvs)
    frame = time_calls(lambda: eng.reconstruct_graphed(views, mvs), args.reps)
    times = {(name, K): [] for name in variants for K in ks}
    for _ in range(args.rounds):
        for K in ks:
            for name, fn in variants.items():
                times[(name, K)].append(time_calls(lambda: fn(K), args.reps))
    res = {"gpu": info, "config": f"{args.depths}x{args.side}x{args.side} steps {args.steps} bf16", "temperature": T,
           "frame_z0_ms": round(frame, 3)}
    print(f"one frame (z = 0, graphed): {frame:.3f} ms")
    print(f"{'K':>3} {'posterior ms':>13} {'multi (mean) ms':>16} {'K singles + torch ms':>21} {'posterior / singles':>20}")
    for K in ks:
        med = {name: statistics.median(times[(name, K)]) for name in variants}
        for name in variants:
            res[f"{name}_K{K}_ms"] = round(med[name], 3)
            res[f"{name}_K{K}_spread_ms"] = round(max(times[(name, K)]) - min(times[(name, K)]), 3)
        print(f"{K:>3} {med['posterior']:>13.3f} {med['multi']:>16.3f} {med['singles']:>21.3f} {med['posterior'] / med['singles']:>20.3f}")
    kn = kernel_numbers(ks, dev)
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
