"""Raw sensor frames -> volumes: what reading the sensor frame directly buys.

1. Kernel: one 2160 x 2160 uint16 frame -> 29 x 512 x 512 normalised bf16 views in the engine's C8 layout, three ways:
   ``LensletLayout.views_c8`` (one pass, csrc/sensor.cu), ``extract_views`` (uint16 read directly) + ``to_c8``, and the route
   the package offered before it read uint16 frames (``frame.float()`` + ``extract_views`` + ``to_c8``).  Each route is captured
   ``--launches`` times into one CUDA graph, with inputs and outputs rotated through buffers larger than the 126 MB L2, and
   timed with CUDA events over the replay.  Bytes are counted from the shapes (window pixels read, views written); GB/s is
   set against the 7.7 TB/s HBM3e figure of the B200 data sheet.
2. End to end at the full 512 x 512 x 96 config: ``StreamingReconstructor`` (depth 2, fp16 host volumes) fed with pinned
   uint16 sensor frames (``sensor=layout``) against pinned fp32 views, ``--frames`` frames per round, the two legs alternated
   in one process for ``--rounds`` rounds each.  Host-to-device bytes per frame are computed from the shapes.
   Under torchrun every rank streams its own frames and the rates are summed over ranks (slowest rank's time).

Prints one JSON line (rank 0) with the GPU name, power limit and SM clock read in the same run; ``--out`` also writes it."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

HBM_TBPS = 7.7
COORDS = [[300 + 370 * (i // 6), 280 + 330 * (i % 6)] for i in range(29)]      # 29 lenslets, 512 x 512 views of a 2160^2 frame


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"error": r.stdout + r.stderr}
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}


def window_pixels(coords, side, H, W):
    """Sensor pixels the views read (the clipped windows of extract_views)."""
    n = 0
    for cy, cx in coords:
        ph = max(min(cy + side // 2, H) - max(cy - side // 2, 0), 0)
        pw = max(min(cx + side // 2, W) - max(cx - side // 2, 0), 0)
        n += ph * pw
    return n


def time_graph(fn, launches: int, reps: int = 5) -> float:
    """Microseconds per launch of ``fn(i)`` captured ``launches`` times into one graph (median over ``reps`` replays)."""
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
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / launches)
    del g
    return statistics.median(ts)


def kernel_leg(dev, launches: int) -> dict:
    from cwfa_b200 import _lib, tc
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.ops import _stream
    H = W = 2160
    S, L = 512, len(COORDS)
    mean, std = 32768.0, 16384.0
    layout = LensletLayout(COORDS, (S, S), mean, std, device=dev)
    n_rot = 16                                                    # 16 x (9.3 MB frame + 16.8 MB C8 + 30.4 MB fp32 views) >> 126 MB L2
    g = torch.Generator().manual_seed(0)
    frames = [torch.randint(0, 65536, (1, 1, H, W), generator=g, dtype=torch.int32).to(torch.uint16).to(dev) for _ in range(n_rot)]
    c8 = [tc.C8.empty(1, L, S, S, dev, "bf16") for _ in range(n_rot)]
    f32 = [torch.empty((1, L, S, S), device=dev) for _ in range(n_rot)]
    img32 = [torch.empty((1, H, W), device=dev) for _ in range(n_rot)]
    coords = layout.coords

    def fused(i):
        k = i % n_rot
        _lib.call("cwfa_extract_views_c8", frames[k].data_ptr(), 2, coords.data_ptr(), c8[k].data.data_ptr(), 1, H, W, L, c8[k].Cp,
                  S, S, mean, std, 1, 1, _stream())

    def two_pass(i, src=None, code=2):
        k = i % n_rot
        img = frames[k] if src is None else src[k]
        _lib.call("cwfa_extract_views", img.data_ptr(), code, coords.data_ptr(), f32[k].data_ptr(), 1, H, W, L, S, S, mean, std, 1,
                  _stream())
        _lib.call("cwfa_nchw_to_c8", f32[k].data_ptr(), c8[k].data.data_ptr(), 1, L, c8[k].Cp, S * S, 1, _stream())

    def float_then_two_pass(i):
        k = i % n_rot
        img32[k].copy_(frames[k].view(1, H, W))                   # frame.float(): the conversion pass
        two_pass(i, img32, 0)

    # correctness of what is timed: all three routes give the same bits
    pix = window_pixels(COORDS, S, H, W)
    c8_bytes = c8[0].Cp * S * S * 2
    views_bytes = L * S * S * 4
    routes = [("extract_views_c8", fused, pix * 2 + c8_bytes),
              ("extract_views+to_c8", two_pass, pix * 2 + views_bytes + views_bytes + c8_bytes),
              ("float+extract_views+to_c8", float_then_two_pass, H * W * (2 + 4) + pix * 4 + views_bytes + views_bytes + c8_bytes)]
    rows, ref = {}, None
    for name, fn, nbytes in routes:
        try:
            fn(0)
        except (RuntimeError, NotImplementedError) as e:        # torch's uint16 -> fp32 copy is not available in every build
            rows[name] = dict(error=f"{type(e).__name__}: {e}")
            continue
        bits = c8[0].data.view(torch.int16).clone()
        ref = bits if ref is None else ref
        us = time_graph(fn, launches)
        rows[name] = dict(us=us, bytes=nbytes, GBps=nbytes / us * 1e-3, share_of_hbm_peak=nbytes / us * 1e-6 / HBM_TBPS,
                          bitwise_equal_to_fused=torch.equal(bits, ref))
    for name, key in (("extract_views+to_c8", "speedup_vs_two_pass"), ("float+extract_views+to_c8", "speedup_vs_float_route")):
        if "us" in rows[name]:
            rows[key] = rows[name]["us"] / rows["extract_views_c8"]["us"]
    return dict(frame="2160x2160 uint16", views="29 x 512 x 512 bf16 C8 (Cp 32), normalised", launches=launches,
                rotation=f"{n_rot} frames / outputs (> 126 MB L2)", **rows)


def e2e_leg(dev, frames_per_round: int, rounds: int, world: int) -> dict:
    import cwfa_b200
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine, StreamingReconstructor
    H = W = 2160
    S, D = 512, 96
    model = cwfa_b200.CWFAModel(seed=0).to(dev)
    eng = CWFAEngine(model, "bf16")
    g = torch.Generator().manual_seed(1)
    mvs = [(0.1 * torch.randn((1, D // 2 ** (n + 1), S, S), generator=g)).to(dev) for n in range(4)] + \
          [(0.1 * torch.randn((1, 6, S, S), generator=g)).to(dev)]
    layout = LensletLayout(COORDS, (S, S), 32768.0, 16384.0, device=dev)
    n_rot = 4
    frames = [torch.randint(0, 65536, (1, 1, H, W), generator=g, dtype=torch.int32).to(torch.uint16).pin_memory() for _ in range(n_rot)]
    views = [layout.views(f.to(dev)).cpu().pin_memory() for f in frames]
    outs = [torch.empty((1, D, S, S), dtype=torch.float16, pin_memory=True) for _ in range(4)]
    legs = {"sensor_uint16": (StreamingReconstructor(eng, tuple(frames[0].shape), mvs, depth=2, out_dtype=torch.float16, sensor=layout,
                                                     frame_dtype=torch.uint16), frames),
            "views_fp32": (StreamingReconstructor(eng, tuple(views[0].shape), mvs, depth=2, out_dtype=torch.float16), views)}
    for st, inp in legs.values():                                 # warm-up (graphs are captured at construction)
        st.run([inp[i % n_rot] for i in range(6)], [outs[i % 4] for i in range(6)])
    torch.cuda.synchronize()
    # the two legs give the same volume for the same frame
    o_s, o_v = torch.empty_like(outs[0]), torch.empty_like(outs[0])
    legs["sensor_uint16"][0].run([frames[1]], [o_s])
    legs["views_fp32"][0].run([views[1]], [o_v])
    same = torch.equal(o_s, o_v)
    fps = {k: [] for k in legs}
    for _ in range(rounds):
        for name, (st, inp) in legs.items():
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st.run([inp[i % n_rot] for i in range(frames_per_round)], [outs[i % 4] for i in range(frames_per_round)])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device=dev)
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
                ms = float(t)
            fps[name].append(world * frames_per_round / ms * 1e3)
    res = dict(config="512x512x96, bf16, StreamingReconstructor depth 2, fp16 host volumes", n_gpus=world,
               frames_per_round=frames_per_round, rounds=rounds, same_volume=same)
    for name, v in fps.items():
        res[name] = dict(frames_per_s_median=statistics.median(v), frames_per_s=v, spread=(max(v) - min(v)) / statistics.median(v),
                         h2d_bytes_per_frame=int(frames[0].numel() * 2 if name == "sensor_uint16" else views[0].numel() * 4))
    res["ratio_sensor_over_views"] = res["sensor_uint16"]["frames_per_s_median"] / res["views_fp32"]["frames_per_s_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--frames", type=int, default=200, help="frames per round and leg (per rank)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_sensor_stream.py: no CUDA device; cwfa_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    res = dict(gpu=gpu_info(local))
    if rank == 0:
        res["kernel"] = kernel_leg(dev, args.launches)
    if not args.no_e2e:
        res["e2e"] = e2e_leg(dev, args.frames, args.rounds, world)
    res["gpu_after"] = gpu_info(local)
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
