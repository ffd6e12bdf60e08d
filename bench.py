#!/usr/bin/env python
"""Benchmark of the CWFA hot path: full 512x512x96 inverse reconstruction (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU implementation on the host cores

Prints ONE JSON line (rank 0).  A "step" is the reconstruction of one frame (batch 1) per GPU.
 value        frames/s with the inputs already resident in HBM (CUDA-event timed, max over ranks)
 e2e          frames/s through the host-buffer API (pinned H2D of the views + D2H of the volume inside the timing)
 roofline     dominant kernel class (tcgen05 convolutions) algorithmic TFLOP/s over its summed launch time vs measured peak
 cpu_baseline the reference itself (oracle/_ref, staged by oracle/make_ref.py; "port" = the oracle if the copy is absent) on the
              SAME frame at full size on the host cores (rank 0, N = 1)
 parity       per-level rel-L2 / max-abs / log-det error of the bf16 AND fp16 engines against that CPU run of the same frame
 extra        module-API frames/s, forward NLL (eager + CUDA graph), DP training step (configs[3]), 1024-frame stream (configs[4])

--dump-outputs DIR writes the volume the last timed step reconstructed (rank 0) to DIR/volume.npy, so that two builds can be
compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cwfa_512x512x96_reconstructions_per_sec"
UNIT = "frames/s"
PUBLISHED_FPS = 1.0 / 0.16          # reference README.md:29 "around 0.16 seconds per frame", hardware not stated
# SURVEY.md 8(d): algorithmic conv flops (2*MAC, true channel counts) of one full inverse frame
FRAME_FLOP = 4.3971e12
# --dump-outputs: an array larger than this many elements is stored as a fixed sample (32 MiB in float32)
DUMP_MAX_ELEMS = 8 << 20


def conv_flops_per_frame(cfg):
    """Algorithmic flops of the convolutions that run on the tensor-core kernel, per frame (2*MAC)."""
    S, D, L = cfg["side"], cfg["depths"], cfg["steps"]
    P = S * S
    total = 0.0
    for n in range(L - 1):
        ch = D // 2 ** (n + 1)
        total += 2.0 * P * (614400 + 5504 * ch)                    # 5 sub-networks (SURVEY 8a4)
        total += 2.0 * P * (9 * 29 * ch * 2 + 9 * ch * ch)         # conditioning net 2-D convs
        total += 2.0 * P * ch * (27 * 32 * 2)                      # depth stencil Conv3d(1,32,3) + Conv3d(32,1,3), true 3-D MACs
    nd = D // 2 ** (L - 1)
    unet = (9 * nd * 256 + 9 * 256 * 256) * P + (9 * 256 * 512 + 9 * 512 * 512) * P / 4 + \
           (9 * 512 * 1024 + 9 * 1024 * 1024) * P / 16 + (4 * 1024 * 512) * P / 16 + (2 * 9 * 512 * 512) * P / 4 + \
           (4 * 512 * 256) * P / 4 + (2 * 9 * 256 * 256) * P + 256 * nd * P + 29 * nd * P
    total += 2.0 * unet
    total += 2.0 * P * (49 * 64 * 64 + 64 * 64)                    # ConvNeXt 7x7 + 1x1 (64 channels)
    return total


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def synthetic_inputs(cfg, device, seed):
    """BASELINE.md section 5: views N(0,1) (1,29,S,S); mean-volume pyramid 0.1*N(0,1); z = 0."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    S, D, L = cfg["side"], cfg["depths"], cfg["steps"]
    views = torch.randn((1, 29, S, S), generator=g)
    mvs = [0.1 * torch.randn((1, D // 2 ** (n + 1), S, S), generator=g) for n in range(L - 1)]
    mvs.append(0.1 * torch.randn((1, D // 2 ** (L - 1), S, S), generator=g))
    return views, mvs


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the only code of this file that touches oracle/): the reference itself when its staged copy is present
# ---------------------------------------------------------------------------------------------------------------------
def reference_available() -> bool:
    from oracle import ref_import
    return ref_import.available()


def run_reference_frames(cfg, threads, steps, warmup, seed=0, state=None, return_levels=False):
    """Times the REFERENCE's inverse reconstruction (its own networks.py / FrEIA modules, CWFA.py:865-924 loop) at the full
    size of ``cfg`` on the host cores.  ``state``: optional (state_dicts, PermuteDim axes) of this repo's model, loaded into the
    reference modules so both arms compute the SAME network.  Returns dict(fps, sec, steps, outs, jacs)."""
    from oracle import ref_import
    torch.set_num_threads(threads)
    S, D, L = cfg["side"], cfg["depths"], cfg["steps"]
    inns, conds, enc = ref_import.build_reference_model(D, S, L, seed=seed, lrnn_size=S)
    if state is not None:
        for n, (isd, csd, axes) in enumerate(state["levels"]):
            inns[n].load_state_dict(isd)
            conds[n].load_state_dict(csd)
            for idx, ax in axes.items():
                inns[n].module_list[idx].dims_to_permute = [1, ax]
        enc.load_state_dict(state["lrnn"])
    enc.train()                                        # the reference's LRNN mode at inference (CWFA.py:531-532): batch-statistics BN
    views, mvs = synthetic_inputs(cfg, "cpu", state["input_seed"] if state is not None else seed)
    ts, outs, jacs = [], {}, {}
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            vol = enc(views, mvs[L - 1])[-1]
            outs[L - 1] = vol
            for n in range(L - 2, -1, -1):
                cond_processed = [conds[n](views)[-1].float(), mvs[n]]
                z = torch.zeros((1,) + tuple(inns[n].global_out_shapes[0]))
                vol, jac = inns[n]([z, vol], c=cond_processed, rev=True)
                outs[n], jacs[n] = vol, jac
            dt = time.perf_counter() - t0
            if i >= warmup:
                ts.append(dt)
    t = sum(ts) / len(ts)
    return dict(fps=1.0 / t, sec=t, steps=len(ts), outs=outs if return_levels else None, jacs=jacs if return_levels else None)


def run_cpu_oracle(cfg, threads, steps, warmup, om, seed, return_levels=False):
    """Fallback when oracle/_ref is absent: the oracle port (oracle/cwfa_oracle.py) on the same frame."""
    from oracle import cwfa_oracle as O
    torch.set_num_threads(threads)
    views, mvs = synthetic_inputs(cfg, "cpu", seed)
    ts = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            outs, jacs = O.reconstruct(om, views, mvs, bn_mode="batch", return_all=True)
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    t = sum(ts) / len(ts)
    return dict(fps=1.0 / t, sec=t, steps=len(ts), outs=outs if return_levels else None, jacs=jacs if return_levels else None)


def bind_to_gpu_numa_node(index: int):
    """Pins this process to the CPUs next to GPU ``index`` so that the pinned host buffers of the end-to-end measurement are
    first-touched on the GPU's own socket (with 8 ranks streaming 130 MB per frame each, buffers that all land on one NUMA node
    make half of the GPUs copy across the socket interconnect).  Sources, in order: NVML's ideal CPU affinity of the device
    (what `nvidia-smi topo -m` prints), then sysfs' numa_node of the PCI function.  Returns (description or None, reason)."""
    allowed = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
    except Exception as ex:
        return None, f"nvml unavailable ({type(ex).__name__}: {ex})"
    try:
        ncpu = os.cpu_count() or 1
        words = (max(allowed | {ncpu - 1}) + 64) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            return f"nvml cpu affinity ({len(use)} cpus)", f"pinned to {len(use)} of {len(allowed)} allowed CPUs (NVML ideal affinity of GPU {index})"
        why = "NVML affinity covers every allowed CPU (single NUMA domain or cpuset already local)" if use else "NVML affinity disjoint from this process' cpuset"
    except Exception as ex:
        why = f"nvmlDeviceGetCpuAffinity failed ({type(ex).__name__})"
    try:
        bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
        bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
        if len(bdf.split(":")[0]) == 8:                  # NVML prints an 8-digit domain; sysfs uses 4
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None, why + f"; sysfs numa_node of {bdf} is {node}"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        use = cpus & allowed
        if not use:
            return None, why + f"; node {node} has no CPU in this process' cpuset"
        os.sched_setaffinity(0, use)
        return f"numa node {node}", f"pinned to {len(use)} CPUs of NUMA node {node} (sysfs)"
    except Exception as ex:
        return None, why + f"; sysfs lookup failed ({type(ex).__name__})"


def dump_outputs(out_dir, arrays):
    """Writes each tensor of ``arrays`` as ``out_dir/<name>.npy`` in float32.  A tensor of more than DUMP_MAX_ELEMS elements is
    stored as the 1-D sample of its flattened values at DUMP_MAX_ELEMS positions drawn without replacement by a generator seeded
    with 0, in increasing order: the positions depend on the shape only, so dumps of two builds compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > DUMP_MAX_ELEMS:
            pos = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            a = a.reshape(-1)[pos]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def pctl(vals, q):
    vals = sorted(vals)
    return vals[min(len(vals) - 1, int(round(q * (len(vals) - 1))))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cwfa_b200", choices=["cwfa_b200", "reference"])
    ap.add_argument("--kind", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--side", type=int, default=512)
    ap.add_argument("--depths", type=int, default=96)
    ap.add_argument("--down-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-nll", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-stream", action="store_true")
    ap.add_argument("--stream", type=int, default=0, help="frames of the configs[4] stream over all ranks (default 128 per rank)")
    ap.add_argument("--out-dtype", default="fp16", choices=["fp32", "fp16"],
                    help="dtype of the volume handed back to the host in the e2e leg (fp16 = what the reference's own GPU path produces under its "
                         "default autocast, CWFA.py:845; the other dtype is measured too and reported in extra)")
    ap.add_argument("--inflight", type=int, default=2, help="graph instances (frames) in flight per GPU")
    ap.add_argument("--e2e-inflight", type=int, default=2, help="frames in flight in the host-buffer streaming measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the volume the last of them reconstructed (rank 0) to DIR/volume.npy "
                         "(float32; a fixed seeded sample of its elements when it is larger than 32 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(side=args.side, depths=args.depths, steps=args.down_steps)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = (f"configs[1]: full CWFA inverse reconstruction {args.side}x{args.side}x{args.depths} from synthetic XLFM views + "
                f"mean-volume prior, batch 1 per GPU, {args.down_steps} steps (4 flow levels + LRNN), z=0, random-init weights")

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = os.cpu_count() or 1
        steps, warmup = max(1, args.steps), max(1, args.warmup)
        if reference_available():
            # the reference's own modules at the FULL size; if K + W full frames do not fit a ~4 minute budget the number of
            # timed frames is reduced (never below 3) and reported
            probe = run_reference_frames(cfg, threads, 1, 1)
            fit = max(3, int(200.0 / probe["sec"]) - 1)
            r = run_reference_frames(cfg, threads, min(steps, fit), min(warmup, 1))
            kind, steps_done = "reference", r["steps"]
            note = ("UNMODIFIED reference (oracle/_ref: networks.py + vendored FrEIA + unet.py, its own constructors and random init, "
                    "driver loop of CWFA.py:865-924 at z = 0), fp32 on the host cores")
            sample = (f"{steps_done} timed full-size frames ({args.side}x{args.side}x{args.depths}, batch 1) after {min(warmup, 1) + 2} untimed, "
                      f"{threads} host threads, {r['sec']:.2f} s per frame" + ("" if steps_done == steps else f" (requested {steps}: capped to fit a few minutes)"))
        else:
            import cwfa_b200
            model = cwfa_b200.CWFAModel(n_depths=args.depths, volume_side_size=args.side, INN_max_down_steps=args.down_steps, seed=0)
            r = run_cpu_oracle(cfg, threads, min(steps, 3), 1, model.export_for_oracle(), 0)
            kind, steps_done = "port", r["steps"]
            note = "oracle port of the reference path (oracle/_ref not staged: run oracle/make_ref.py where /root/reference exists)"
            sample = f"{steps_done} timed full-size frames, CPU oracle fp32, {threads} threads, {r['sec']:.2f} s per frame"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": r["fps"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps_done, "warmup": min(warmup, 1) + (2 if kind == "reference" else 0),
            "ms_per_step": r["sec"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": r["fps"] / PUBLISHED_FPS, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload, "note": note},
            "cpu_baseline": {"value": r["fps"], "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": r["fps"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------ CUDA arm
    import cwfa_b200
    from cwfa_b200 import _lib, tc
    from cwfa_b200.engine import CWFAEngine, StreamingReconstructor
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; cwfa_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa, numa_why = bind_to_gpu_numa_node(local_rank) if world > 1 else (None, "single process: not pinned")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    _lib.call("cwfa_device_check")

    model = cwfa_b200.CWFAModel(n_depths=args.depths, volume_side_size=args.side, INN_max_down_steps=args.down_steps, seed=0).to(dev)
    eng = CWFAEngine(model, args.kind)
    n_rot = 4                                               # rotate device-resident inputs between steps
    inputs = [synthetic_inputs(cfg, dev, 100 + rank * 16 + i) for i in range(n_rot)]
    views_dev = [v.to(dev) for v, _ in inputs]
    mvs_dev = [m.to(dev) for m in inputs[0][1]]             # dataset constants (mean-volume pyramid), replicated
    views_host = [v.pin_memory() for v, _ in inputs]        # allocated AFTER the NUMA pin: first-touched on the GPU's socket

    # launches per step, counted on one eager pass (the graph replays exactly these launches)
    c0 = _lib.launch_count
    eng.reconstruct(views_dev[0], mvs_dev)
    launches_per_step = _lib.launch_count - c0
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput: a stream of frames whose inputs are already in HBM; `depth` graph instances in
    # flight (frames are independent; consecutive frames overlap on the GPU), outputs written to device buffers
    depth = 1 if args.no_graph else args.inflight
    streamer = StreamingReconstructor(eng, tuple(views_dev[0].shape), mvs_dev, depth=depth) if not args.no_graph else None
    outs_dev = [torch.empty((1, args.depths, args.side, args.side), device=dev, dtype=torch.float32) for _ in range(2)]

    def run_frames(k):
        """Reconstructs k frames; returns the volume of the last one."""
        if streamer is None:
            for i in range(k):
                last = eng.reconstruct(views_dev[i % n_rot], mvs_dev)
            return last
        streamer.run([views_dev[i % n_rot] for i in range(k)], [outs_dev[i % 2] for i in range(k)])
        return outs_dev[(k - 1) % 2]

    run_frames(max(3, args.warmup))
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    last_volume = run_frames(args.steps)
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"volume": last_volume})
    del last_volume
    # single-stream, one-graph-at-a-time latency of a frame (reported next to the throughput)
    if streamer is not None:
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record()
        for i in range(5):
            eng.reconstruct_graphed(views_dev[i % n_rot], mvs_dev)
        l1.record()
        torch.cuda.synchronize()
        frame_latency_ms = l0.elapsed_time(l1) / 5
    else:
        frame_latency_ms = elapsed_ms / args.steps

    # ---- end to end through the host-buffer streaming API: every step copies its views H2D from pinned memory and
    # its reconstructed volume D2H into pinned memory; copies of neighbouring frames overlap the compute
    out_dt = torch.float16 if args.out_dtype == "fp16" else torch.float32
    streamer_h = StreamingReconstructor(eng, tuple(views_host[0].shape), mvs_dev, depth=args.e2e_inflight, out_dtype=out_dt)
    outs_host = [torch.empty((1, args.depths, args.side, args.side), dtype=out_dt, pin_memory=True) for _ in range(4)]
    streamer_h.run([views_host[i % n_rot] for i in range(3)], [outs_host[i % 4] for i in range(3)])
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e2.record()
    streamer_h.run([views_host[i % n_rot] for i in range(args.steps)], [outs_host[i % 4] for i in range(args.steps)])
    e3.record()
    barrier()
    e2e_ms = e2.elapsed_time(e3)
    e2e_host_ms = (time.perf_counter() - t_host0) * 1e3      # host wall clock around the same region (sanity)
    # the same with the OTHER host dtype of the volume (fp32: 100.7 MB D2H per frame, fp16: 50.3 MB) -- reported in extra
    other = "fp32" if args.out_dtype == "fp16" else "fp16"
    e2e_other_ms = None
    try:
        odt = torch.float32 if other == "fp32" else torch.float16
        st_o = StreamingReconstructor(eng, tuple(views_host[0].shape), mvs_dev, depth=args.e2e_inflight, out_dtype=odt)
        outs_o = [torch.empty((1, args.depths, args.side, args.side), dtype=odt, pin_memory=True) for _ in range(4)]
        st_o.run([views_host[i % n_rot] for i in range(3)], [outs_o[i % 4] for i in range(3)])
        barrier()
        h0_, h1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0_.record()
        st_o.run([views_host[i % n_rot] for i in range(args.steps)], [outs_o[i % 4] for i in range(args.steps)])
        h1_.record()
        barrier()
        e2e_other_ms = h0_.elapsed_time(h1_)
        # copy-only ceiling for THAT dtype's traffic as well
        so_a, so_b = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        sti, sto = torch.empty_like(views_dev[0]), torch.empty((1, args.depths, args.side, args.side), device=dev, dtype=odt)
        c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0_.record()
        for i in range(args.steps):
            with torch.cuda.stream(so_a):
                sti.copy_(views_host[i % n_rot], non_blocking=True)
            with torch.cuda.stream(so_b):
                outs_o[i % 4].copy_(sto, non_blocking=True)
        torch.cuda.current_stream().wait_stream(so_a)
        torch.cuda.current_stream().wait_stream(so_b)
        c1_.record()
        barrier()
        copy_other_ms = c0_.elapsed_time(c1_)
        del st_o, outs_o, sti, sto
    except Exception as ex:
        copy_other_ms = None
        print(f"bench: {other}-volume e2e leg failed: {ex!r}", file=sys.stderr)
    # copy-only ceiling of the same host traffic (no compute): what the platform allows for these bytes per frame
    cp0, cp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st_in, st_out = torch.empty_like(views_dev[0]), torch.empty((1, args.depths, args.side, args.side), device=dev, dtype=out_dt)
    s_a, s_b = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    barrier()
    cp0.record()
    for i in range(args.steps):
        with torch.cuda.stream(s_a):
            st_in.copy_(views_host[i % n_rot], non_blocking=True)
        with torch.cuda.stream(s_b):
            outs_host[i % 4].copy_(st_out, non_blocking=True)
    torch.cuda.current_stream().wait_stream(s_a)
    torch.cuda.current_stream().wait_stream(s_b)
    cp1.record()
    barrier()
    copy_only_ms = cp0.elapsed_time(cp1)
    # single-frame latency through the synchronous host call (reported, not the throughput headline)
    out_host32 = torch.empty((1, args.depths, args.side, args.side), dtype=torch.float32, pin_memory=True)
    lat0 = time.perf_counter()
    eng.reconstruct_host(views_host[0], mvs_dev, out_host32)
    eng.reconstruct_host(views_host[1], mvs_dev, out_host32)
    sync_latency_ms = (time.perf_counter() - lat0) * 1e3 / 2
    clocks = sampler.stop() if rank == 0 else None
    del streamer_h

    if world > 1:
        t = torch.tensor([elapsed_ms, e2e_ms, copy_only_ms, e2e_other_ms or 0.0, copy_other_ms or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms, copy_only_ms = float(t[0]), float(t[1]), float(t[2])
        e2e_other_ms = float(t[3]) if e2e_other_ms else None
        copy_other_ms = float(t[4]) if copy_other_ms else None

    # ---- dominant-kernel roofline: sum of tcgen05 conv launch durations over one step (CUDA events on the launch stream)
    conv_ms, n_conv, per_kernel = 0.0, 0, {}
    if rank == 0:
        evs = []
        orig = _lib.call

        def timed_call(name, *a):
            if name in ("cwfa_conv_tc", "cwfa_conv_tc_bn", "cwfa_resblock_tc", "cwfa_resblock_tc_batched", "cwfa_conv_tc_coupling", "cwfa_coupling_tc", "cwfa_coupling_f8", "cwfa_stencil3d_tc"):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                orig(name, *a)
                e.record()
                evs.append((name, s, e))
            else:
                orig(name, *a)

        _lib.call = timed_call
        tc._lib.call = timed_call
        try:
            for rep in range(2):                 # first pass warms, second is measured
                evs.clear()
                eng.reconstruct(views_dev[1], mvs_dev)
                torch.cuda.synchronize()
        finally:
            _lib.call = orig
        for name, s, e in evs:
            d = s.elapsed_time(e)
            conv_ms += d
            k = per_kernel.setdefault(name, [0, 0.0])
            k[0] += 1
            k[1] += d
        n_conv = len(evs)

    # ---- the drop-in MODULE API with the tensor-core switch (cwfa_b200.set_inference_precision): the calls the reference
    # itself makes (cond_nets[n](views), conv_inn[n]([z, vol], c=..., rev=True), CWFA.py:882-912), eager, device-resident inputs
    module_fps = None
    if rank == 0:
        with cwfa_b200.inference_precision(args.kind):
            for i in range(3):
                model.reconstruct(views_dev[i % n_rot], mvs_dev)
            torch.cuda.synchronize()
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nm = 10
            m0.record()
            for i in range(nm):
                model.reconstruct(views_dev[i % n_rot], mvs_dev)
            m1.record()
            torch.cuda.synchronize()
        module_fps = nm / (m0.elapsed_time(m1) * 1e-3)

    # ---- secondary metric of BASELINE.json: forward pass + per-level NLL / log-det (configs[2], batch 8): eager and CUDA graph
    nll_fps = nll_graph_fps = None
    if rank == 0 and not args.no_nll:
        B = 8
        g = torch.Generator(device="cpu").manual_seed(7)
        vol = torch.randn((B, args.depths, args.side, args.side), generator=g).to(dev)
        vB = torch.randn((B, 29, args.side, args.side), generator=g).to(dev)
        mvB = [m.repeat(B, 1, 1, 1) for m in mvs_dev[:model.n_levels]]

        def median_of(fn, reps=3):
            times = []
            for _ in range(reps):
                n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n0.record()
                fn()
                n1.record()
                torch.cuda.synchronize()
                times.append(n0.elapsed_time(n1))
            return sorted(times)[len(times) // 2]

        for _ in range(2):                          # warm-up: allocator pools for the batch-8 activations, kernel loading
            eng.forward_nll(vol, vB, mvB)
        torch.cuda.synchronize()
        nll_fps = B / (median_of(lambda: eng.forward_nll(vol, vB, mvB)) * 1e-3)
        try:
            eng.forward_nll_graphed(vol, vB, mvB)
            torch.cuda.synchronize()
            nll_graph_fps = B / (median_of(lambda: eng.forward_nll_graphed(vol, vB, mvB), 5) * 1e-3)
        except Exception as ex:
            nll_graph_fps = None
            print(f"bench: graphed forward NLL failed: {ex!r}", file=sys.stderr)
        eng._graphs = {k: v for k, v in eng._graphs.items() if k[0] != "nll"}
        del vol, vB, mvB
        torch.cuda.empty_cache()

    # ---- BASELINE.json configs[4]: streaming reconstruction of seeded frames (seed = frame id) sharded over the ranks,
    # batch sweep; frames/s over all ranks (max-over-ranks time) and rank 0's per-frame in-pipeline latency percentiles
    stream_rows, stream_err = [], None
    if not args.no_stream and not args.no_graph:
        try:
            from cwfa_b200.sharding import frame_seed, frame_shard
            total = args.stream if args.stream > 0 else 128 * world
            a, b = frame_shard(total, rank, world)
            frames = [torch.randn((1, 29, args.side, args.side), generator=torch.Generator().manual_seed(frame_seed(f))).to(dev) for f in range(a, b)]
            for Bs in (1, 2, 4, 8, 16):
                if len(frames) < 3 * Bs:
                    continue
                mvb = [m.repeat(Bs, 1, 1, 1) for m in mvs_dev]
                batches = [torch.cat(frames[i:i + Bs]) for i in range(0, len(frames) - Bs + 1, Bs)]
                st = StreamingReconstructor(eng, tuple(batches[0].shape), mvb, depth=2)
                outs = [torch.empty((Bs, args.depths, args.side, args.side), device=dev) for _ in range(3)]
                st.run(batches[:3], outs[:3])
                lat = []
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                barrier()
                s0.record()
                st.run(batches, [outs[i % 3] for i in range(len(batches))], latency_events=lat)
                s1.record()
                barrier()
                ms = s0.elapsed_time(s1)
                nfr = torch.tensor([ms, float(len(batches) * Bs)], device=dev, dtype=torch.float64)
                if world > 1:
                    tmax = nfr[:1].clone()
                    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                    tot = nfr[1:].clone()
                    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
                    ms, n_all = float(tmax), float(tot)
                else:
                    n_all = float(nfr[1])
                ls = [s.elapsed_time(e) for s, e in lat]
                stream_rows.append(dict(batch=Bs, frames=int(n_all), frames_per_s=n_all / ms * 1e3, latency_ms_p50=pctl(ls, 0.5),
                                        latency_ms_p99=pctl(ls, 0.99)))
                del st, outs, batches, mvb
                eng._graphs = {k: v for k, v in eng._graphs.items() if k[0][0] == 1}      # keep only the batch-1 frame graphs
                torch.cuda.empty_cache()
            del frames
        except Exception as ex:
            stream_err = repr(ex)[:200]

    # ---- CPU leg + parity (rank 0, N = 1): the reference itself (or the oracle port) on frame 0 with THIS model's weights
    cpu_baseline = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        try:
            from cwfa_b200.modules import PermuteDim
            cpu = lambda sd: {k: v.detach().cpu().clone() for k, v in sd.items()}
            if reference_available():
                state = dict(levels=[(cpu(model.conv_inn[n].state_dict()), cpu(model.cond_nets[n].state_dict()),
                                      {i: m.axis for i, m in enumerate(model.conv_inn[n].module_list) if isinstance(m, PermuteDim)})
                                     for n in range(model.n_levels)], lrnn=cpu(model.cond_nets[-1].state_dict()), input_seed=100)
                r = run_reference_frames(cfg, threads, 2, 1, state=state, return_levels=True)
                kind_cpu = "reference"
                how = "the UNMODIFIED reference (oracle/_ref: networks.py + FrEIA, loaded with this model's state_dicts)"
            else:
                r = run_cpu_oracle(cfg, threads, 2, 1, model.export_for_oracle(), 100, return_levels=True)
                kind_cpu = "port"
                how = "the oracle port (oracle/_ref not staged)"
            cpu_baseline = {"value": r["fps"], "unit": UNIT, "cores": threads, "kind": kind_cpu,
                            "sample": f"{r['steps']} timed steps (after 1 warm-up) of the SAME workload at full size ({args.side}x{args.side}x{args.depths}, "
                                      f"batch 1, frame seed 100), {how}, fp32, {threads} threads, {r['sec']:.1f} s per frame"}
            # parity of both engine precisions against that CPU run of the same frame, per level (BASELINE.json: "max-abs err")
            parity = {"against": kind_cpu, "frame_seed": 100, "levels": "index L-1 = LRNN output, 0 = full volume"}
            v0 = synthetic_inputs(cfg, "cpu", 100)[0].to(dev)
            for kd in ("bf16", "fp16"):
                e_ = eng if kd == args.kind else CWFAEngine(model, kd)
                outs, jacs = e_.reconstruct(v0, mvs_dev, return_all=True)
                rows = {}
                for n in sorted(outs):
                    ref = r["outs"][n].double()
                    got = outs[n].double().cpu()
                    row = {"rel_l2": float((got - ref).norm() / ref.norm()), "max_abs": float((got - ref).abs().max()),
                           "ref_abs_max": float(ref.abs().max())}
                    if n in jacs:
                        rj = float(r["jacs"][n][0])
                        row["logdet_rel_err"] = abs(float(jacs[n][0]) - rj) / max(abs(rj), 1e-30)
                    rows[str(n)] = row
                parity[kd] = rows
                del outs, jacs
        except Exception as ex:
            cpu_baseline = cpu_baseline or {"error": repr(ex)[:300]}
            parity = parity or {"error": repr(ex)[:300]}

    # ---- BASELINE.json configs[3]: data-parallel training step (one frame per rank): flow level 0 (forward NLL + inverse MSE +
    # backward + gradient all-reduce + Lion) and the LRNN step, tensor-core convolutions; all ranks take part
    train = {}
    if not args.no_train:
        try:
            from cwfa_b200.training import FlowLevelTrainer, LRNNTrainer
            g = torch.Generator(device="cpu").manual_seed(11 + rank)
            C = args.depths
            mk = lambda ch, sc=1.0: (torch.randn((1, ch, args.side, args.side), generator=g) * sc).to(dev)
            gt, vw, mv0, vin = mk(C), mk(29), mk(C // 2, 0.1), mk(C // 2)
            tr = FlowLevelTrainer(model, 0, precision=args.kind)

            def timed(fn, warm, reps):
                for _ in range(warm):
                    fn()
                barrier()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(reps):
                    fn()
                t1.record()
                barrier()
                ms = torch.tensor([t0.elapsed_time(t1) / reps], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                return float(ms)

            ms0 = timed(lambda: tr.step(gt, vw, mv0, vin), 2, 5)
            train.update(level0_ms_per_step=ms0, level0_frames_per_s=world * 1000.0 / ms0, level0_collectives_per_step=tr.collectives,
                         level0_allreduce_bytes=int(sum(g_.numel() for o in (tr.optimizer, tr.optimizer_cond) for g_ in o.flat_grads()) * 4))
            tr.release()
            if world == 1:            # the same step captured as ONE CUDA graph (trainer graph=True; eager under data parallelism)
                trg = FlowLevelTrainer(model, 0, precision=args.kind, graph=True)
                train.update(level0_graph_ms_per_step=timed(lambda: trg.step(gt, vw, mv0, vin), 2, 5))
                trg.release()
                del trg
            del tr, gt, mv0, vin
            nd = C // 2 ** (args.down_steps - 1)
            gt_l = mk(nd)
            lt = LRNNTrainer(model, precision=args.kind)
            ms1 = timed(lambda: lt.step(gt_l, vw), 2, 3)
            train.update(lrnn_ms_per_step=ms1, lrnn_frames_per_s=world * 1000.0 / ms1, lrnn_collectives_per_step=lt.collectives,
                         lrnn_allreduce_bytes=int(sum(g_.numel() for g_ in lt.optimizer.flat_grads()) * 4))
            lt.release()
            if world == 1:
                ltg = LRNNTrainer(model, precision=args.kind, graph=True)
                train.update(lrnn_graph_ms_per_step=timed(lambda: ltg.step(gt_l, vw), 2, 3))
                ltg.release()
                del ltg
            del lt, gt_l, vw
            torch.cuda.empty_cache()
        except Exception as ex:       # a secondary figure must never take the headline line down
            train["error"] = repr(ex)[:300]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md, sustained ~1.4 PFLOP/s)"
    conv_flop = conv_flops_per_frame(cfg)
    achieved = conv_flop / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else None
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "conv_tc_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        pass
    fps = world * args.steps / (elapsed_ms * 1e-3)
    e2e_fps = world * args.steps / (e2e_ms * 1e-3)
    out_bytes = args.depths * args.side * args.side * (2 if args.out_dtype == "fp16" else 4)
    out = {
        "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": fps / PUBLISHED_FPS, "dtype": args.kind, "data": "synthetic",
        "config": {"workload": workload, "frames_per_gpu_per_step": 1, "sharding": f"frames (1 per rank, {world} ranks), no data-path collective",
                   "rank0_numa_node": numa, "rank0_numa_note": numa_why,
                   "cuda_graph": not args.no_graph, "frames_in_flight": depth, "single_frame_latency_ms": frame_latency_ms,
                   "l2_policy": "per-step working set (activations ~3 GB) exceeds the 126 MB L2; inputs rotate over 4 buffers",
                   "baseline_note": "README.md:29 publishes ~0.16 s/frame on unstated hardware"},
        "clocks": clocks,
        "extra": {f"e2e_{other}_volume_frames_per_s": (world * args.steps / (e2e_other_ms * 1e-3)) if e2e_other_ms else None,
                  f"e2e_{other}_volume_copy_only_frames_per_s": (world * args.steps / (copy_other_ms * 1e-3)) if copy_other_ms else None,
                  "e2e_volume_dtype_note": f"the headline e2e hands the volume back as {args.out_dtype} (fp16 = the reference's own GPU output under its default autocast, CWFA.py:845, "
                                           "narrowed by one cast kernel on the device: 30.4 MB H2D + 50.3 MB D2H per frame); the other dtype (fp32: 100.7 MB D2H) and the "
                                           "copy-only ceiling of its traffic are measured in the same run: at 8 GPUs the fp32 volume is bound by the box's host-side copy rate",
                  "module_api_frames_per_s": module_fps,
                  "module_api_note": "the reference's own entry points (cond_nets[n](views), conv_inn[n]([z, vol], c=..., rev=True)) on this package's drop-in modules with "
                                     f"set_inference_precision('{args.kind}'): eager, device-resident inputs, 10 frames, 1 GPU",
                  "forward_nll_frames_per_s_batch8": nll_fps, "forward_nll_graph_frames_per_s_batch8": nll_graph_fps,
                  "forward_nll_note": "BASELINE.json configs[2]: 4-level forward pyramid + per-level log-det / sum z^2 / NLL, batch 8, 1 GPU; eager and as one CUDA-graph replay (levels as parallel branches)",
                  "train": train,
                  "train_note": "BASELINE.json configs[3]: one frame per rank; flow level 0 (96 -> 48+48 ch): forward NLL + inverse MSE + backward + gradient all-reduce (NCCL) + Lion; "
                                "LRNN step likewise; tensor-core convs (fwd, dgrad, wgrad); frames/s = ranks / max-over-ranks step time; *_graph_ms_per_step (1 GPU): the same "
                                "step captured as ONE CUDA graph (trainer graph=True, bit-identical to the eager steps)",
                  "stream": stream_rows, "stream_error": stream_err,
                  "stream_note": "BASELINE.json configs[4]: frames with seed = frame id sharded contiguously over the ranks (128 per rank unless --stream), 2 graph instances in flight, "
                                 "batch = frames per graph replay; latency = input copy issued -> output written (rank 0, CUDA events)"},
        "e2e": {"value": e2e_fps, "unit": UNIT, "h2d_bytes_per_step": views_host[0].numel() * 4, "d2h_bytes_per_step": out_bytes,
                "ms_per_step": e2e_ms / args.steps, "api": f"StreamingReconstructor.run ({args.e2e_inflight} frames in flight, host volume dtype {args.out_dtype})",
                "sync_call_latency_ms": sync_latency_ms, "host_wall_ms_per_step": e2e_host_ms / args.steps,
                "copy_only_frames_per_s": world * args.steps / (copy_only_ms * 1e-3),
                "copy_only_note": "the same H2D + D2H bytes per frame with NO compute (both directions concurrently): the platform ceiling for this host traffic"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel + resblock_tc_kernel + coupling_f8_kernel + stencil3d_tc_kernel (all tcgen05 implicit-GEMM convolution launches of a frame)", "achieved": achieved, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic,
                     "launches_per_step": n_conv, "avg_launch_us": (conv_ms * 1e3 / n_conv) if n_conv else None,
                     "algorithmic_flop_per_step": conv_flop, "conv_ms_per_step": conv_ms, "peak_source": peak_src,
                     "per_kernel_ms": {k: {"launches": v[0], "ms": v[1]} for k, v in per_kernel.items()},
                     "whole_step_tflops": FRAME_FLOP * (args.side / 512.0) ** 2 / (elapsed_ms / args.steps * 1e-3) / 1e12},
    }
    if cpu_baseline is not None:
        out["cpu_baseline"] = cpu_baseline
    if parity is not None:
        out["parity"] = parity
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
