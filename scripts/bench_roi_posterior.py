"""Cost of the exact posterior mean and std of ROI readouts (``CWFAEngine.roi_posterior_exact_graphed``) at the full configuration
(96 x 512 x 512, 5 steps, bf16, seeded synthetic inputs as bench.py builds them), temperature 0.7, with seeded synthetic
neuron-like ROIs: small ellipsoids (lateral radius 2-4 pixels, 1-3 planes deep), given as a label volume, R = 1000 and 20000.

  * end to end, graphed, alternated within each of ``--rounds`` rounds (same process, same inputs; every timed window ends in a
    device synchronise), batch 1 and ``--batch``: ``reconstruct_graphed``, ``reconstruct_posterior_exact_graphed`` and
    ``roi_posterior_exact_graphed`` at each R;
  * the readout kernel alone (``tc.roi_readout_f8`` on one frame's volume and scale tensors), CUDA events over a graph of
    back-to-back launches, with its table entries and the bytes its walk reads;
  * the ``RoiSet.from_labels`` build time (tables on the CPU, copy to the device);
  * ``sqrt(sum w^2 std^2)`` from the per-voxel exact std against the exact ROI std on the same ROIs: what ignoring the
    correlation between voxels does.

Prints the GPU name, power limit and SM clock read in the same run, then one JSON line; ``--out`` also writes the JSON."""
import argparse
import json
import math
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bench_posterior import gpu_info, synthetic_inputs, time_calls, time_graph


def neuron_labels(D, H, W, R, seed):
    """(D, H, W) int32 labels of R ellipsoids at seeded random centres; a later ROI overwrites an earlier one where they meet."""
    rs = np.random.RandomState(seed)
    lab = np.zeros((D, H, W), dtype=np.int32)
    for r in range(R):
        ry, rx, rz = rs.uniform(2.0, 4.0), rs.uniform(2.0, 4.0), rs.uniform(0.5, 1.5)
        cz, cy, cx = rs.uniform(0, D - 1), rs.uniform(0, H - 1), rs.uniform(0, W - 1)
        z0, z1 = max(0, math.floor(cz - rz)), min(D, math.ceil(cz + rz) + 1)
        y0, y1 = max(0, math.floor(cy - ry)), min(H, math.ceil(cy + ry) + 1)
        x0, x1 = max(0, math.floor(cx - rx)), min(W, math.ceil(cx + rx) + 1)
        z, y, x = np.ogrid[z0:z1, y0:y1, x0:x1]
        m = ((z - cz) / rz) ** 2 + ((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2 <= 1.0
        if not m.any():
            m[round(cz) - z0, round(cy) - y0, round(cx) - x0] = True
        lab[z0:z1, y0:y1, x0:x1][m] = r + 1
    return lab


def naive_std(rs, std):
    """sqrt(sum_v w_v^2 std_v^2) per (b, roi) from the per-voxel exact std (B, D, H, W), float64: the readout std if the voxels
    were independent."""
    B = std.shape[0]
    cnt = (rs.mean_ptr[1:] - rs.mean_ptr[:-1])
    roi = torch.repeat_interleave(torch.arange(rs.n_rois, device=std.device), cnt)
    n = rs.n_mean_entries
    w2 = rs.mean_w[:n].double() ** 2
    out = torch.zeros((B, rs.n_rois), device=std.device, dtype=torch.float64)
    for b in range(B):
        out[b].index_add_(0, roi, w2 * std[b].reshape(-1)[rs.mean_idx[:n].long()].double() ** 2)
    return out.sqrt()


def planes_per_column(rs):
    """Per ROI, the largest number of its voxels in one pixel column: voxels of different columns depend on disjoint latents, so
    only ROIs that span several planes of a column have correlated voxels."""
    S = rs.volume_shape[1] * rs.volume_shape[2]
    cnt = (rs.mean_ptr[1:] - rs.mean_ptr[:-1])
    roi = torch.repeat_interleave(torch.arange(rs.n_rois, device=cnt.device), cnt)
    key = roi * S + rs.mean_idx[:rs.n_mean_entries].long() % S
    k, c = torch.unique(key, return_counts=True)
    out = torch.zeros(rs.n_rois, dtype=torch.int64, device=cnt.device)
    return out.scatter_reduce_(0, k // S, c, reduce="amax")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--depths", type=int, default=96)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--temperature", type=float, default=0.7)
    ap.add_argument("--rois", type=int, nargs="+", default=[1000, 20000])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_roi_posterior.py needs a CUDA device")
    import cwfa_b200
    from cwfa_b200 import tc
    from cwfa_b200.engine import CWFAEngine
    from cwfa_b200.pipeline import truncated_normal_var
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    print("GPU:", info, flush=True)
    T, B, D, S = args.temperature, args.batch, args.depths, args.side
    model = cwfa_b200.CWFAModel(n_depths=D, volume_side_size=S, INN_max_down_steps=args.steps, seed=0).to(dev)
    eng = CWFAEngine(model, "bf16")
    views, mvs = synthetic_inputs(S, D, args.steps)
    views, mvs = views.to(dev), [m.to(dev) for m in mvs]
    g = torch.Generator().manual_seed(1)
    vB = torch.cat([views] + [torch.randn(tuple(views.shape), generator=g).to(dev) for _ in range(B - 1)])
    mvB = [m.repeat(B, 1, 1, 1) for m in mvs]
    res = {"gpu": info, "config": f"{D}x{S}x{S} steps {args.steps} bf16, graphed, temperature {T}"}

    sets = {}
    for R in args.rois:
        lab = neuron_labels(D, S, S, R, 100 + R)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rs = cwfa_b200.RoiSet.from_labels(lab, model.n_levels, device=dev)
        torch.cuda.synchronize()
        res[f"R{R}_build_s"] = round(time.perf_counter() - t0, 3)
        res[f"R{R}_voxels"] = rs.n_mean_entries
        res[f"R{R}_entries"] = rs.n_entries
        sets[R] = rs
        print(f"R = {R}: {rs.n_mean_entries} voxels, {rs.n_entries} table entries, built in {res[f'R{R}_build_s']} s", flush=True)

    variants = {"b1_reconstruct": lambda: eng.reconstruct_graphed(views, mvs),
                "b1_exact": lambda: eng.reconstruct_posterior_exact_graphed(views, mvs, temperature=T)}
    for R, rs in sets.items():
        variants[f"b1_roi_R{R}"] = lambda rs=rs: eng.roi_posterior_exact_graphed(views, mvs, rs, temperature=T)
    variants[f"b{B}_reconstruct"] = lambda: eng.reconstruct_graphed(vB, mvB)
    variants[f"b{B}_exact"] = lambda: eng.reconstruct_posterior_exact_graphed(vB, mvB, temperature=T)
    for R, rs in sets.items():
        variants[f"b{B}_roi_R{R}"] = lambda rs=rs: eng.roi_posterior_exact_graphed(vB, mvB, rs, temperature=T)
    for fn in variants.values():                               # capture and warm every graph before timing
        fn()
        fn()
    times = {name: [] for name in variants}
    for _ in range(args.rounds):
        for name, fn in variants.items():
            times[name].append(time_calls(fn, args.reps))
    for name in variants:
        med = statistics.median(times[name])
        res[f"{name}_ms_per_call"] = round(med, 3)
        res[f"{name}_rounds_ms"] = [round(t, 3) for t in times[name]]
        print(f"{name:>20}: {med:.3f} ms per call  (rounds {res[f'{name}_rounds_ms']})")
    for bb in (1, B):
        for R in sets:
            res[f"b{bb}_roi_R{R}_over_exact"] = round(res[f"b{bb}_roi_R{R}_ms_per_call"] / res[f"b{bb}_exact_ms_per_call"], 4)
            res[f"b{bb}_roi_R{R}_over_reconstruct"] = round(res[f"b{bb}_roi_R{R}_ms_per_call"] / res[f"b{bb}_reconstruct_ms_per_call"], 4)

    # the readout kernel alone, on one batch's volume and scale tensors
    sigma = math.sqrt(truncated_normal_var(T))
    with torch.no_grad():
        for bb, (v_, m_) in ((1, (views, mvs)), (B, (vB, mvB))):
            vol, levels = eng._scale_pass(v_, m_, None, None)
            for hi8, _ in levels:
                vol = tc.haar1d_merge_f8(vol, hi8)
            scales = [sc8 for _, sc8 in reversed(levels)]
            for R, rs in sets.items():
                us = time_graph(lambda: tc.roi_readout_f8(vol, scales, rs, sigma), 20)
                nbytes = bb * 12 * rs.n_entries                # per entry: index, weight / coefficient, gathered value
                res[f"b{bb}_readout_R{R}_us"] = round(us, 2)
                res[f"b{bb}_readout_R{R}_bytes"] = nbytes
                res[f"b{bb}_readout_R{R}_TBps"] = round(nbytes / us / 1e6, 3)
                print(f"readout kernel b{bb} R={R}: {us:.2f} us, {nbytes / 1e6:.1f} MB walked ({nbytes / us / 1e6:.2f} TB/s)")
            del vol, levels, scales

        # what ignoring the voxels' correlation does: sqrt(sum w^2 std^2) against the exact ROI std, frame 0
        _, pstd = eng.reconstruct_posterior_exact(views, mvs, temperature=T)
        for R, rs in sets.items():
            _, _, exact = eng.roi_posterior_exact(views, mvs, rs, temperature=T)
            ok = exact[0] > 0
            ratio = (naive_std(rs, pstd)[0][ok] / exact[0][ok].double()).cpu()
            q = torch.quantile(ratio, torch.tensor([0.05, 0.5, 0.95], dtype=torch.float64)).tolist()
            res[f"R{R}_naive_over_exact_p05_p50_p95"] = [round(x, 4) for x in q]
            res[f"R{R}_naive_over_exact_min_max"] = [round(float(ratio.min()), 4), round(float(ratio.max()), 4)]
            res[f"R{R}_naive_off_by_over_1pct"] = round(float(((ratio - 1).abs() > 0.01).double().mean()), 4)
            res[f"R{R}_multi_plane"] = round(float((planes_per_column(rs) > 1).double().mean()), 4)
            print(f"R = {R}: naive / exact std quantiles 5/50/95 % {q}, min {float(ratio.min()):.4f}, max {float(ratio.max()):.4f}")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
