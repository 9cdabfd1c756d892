#!/usr/bin/env python
"""bench.py -- frames/s on the paris-30k-like scene at 4096x4096 MSAA16 (BASELINE.json configs[2]) and the
fine-stage HBM roofline, next to the CPU baseline (the oracle = restated reference CPU shaders).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W          (one rank per GPU, tile-row stripes assembled over NVLink)
    python bench.py --impl reference ...                (the CPU arm: oracle on the host cores)
    python bench.py ... --dump-outputs DIR              (also write the last timed frame to DIR, see dump_outputs)

One step = one frame of the hot path (pathtag .. fine) over the synthetic scene; --steps is the number of timed steps.
`value`  : frames/s with the packed scene already resident in HBM (vb_render_resident).
`e2e`    : frames/s through the C ABI with pinned HOST buffers (streaming `vb_render_begin`; the blocking one-call
           `vb_render` figure is reported next to it): scene H2D + render +
           full image D2H inside the timed region.
Timing   : CUDA events on the renderer's stream around every step; L2 is flushed (256 MiB write) between
           steps outside the event pairs; max over ranks; clocks sampled with nvidia-smi during the run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(name="paris-like-30k 4096x4096 MSAA16", n_paths=30000, size=4096, seed=30000, aa=2)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def build_scene(args):
    from vello_b200 import scenes
    from vello_b200.encoding import resolve
    t = time.time()
    if args.scene == "tiger":        # BASELINE.json configs[1]: tiger at args.size x args.height
        sc = scenes.tiger(args.size, args.height or args.size)
    elif args.scene == "beziers":    # configs[4]: cubic paths + nested clips
        sc = scenes.beziers_clips(args.paths, max(1, args.paths // 100), args.size, seed=100000)
    else:                            # configs[2] (default, the headline workload)
        sc = scenes.paris_like(args.paths, args.size, args.seed)
    packed = resolve(sc.encoding)
    return packed, time.time() - t


DUMP_BYTES = 48 << 20  # float32 pixels per dump: with the row indices, a dump stays below 64 MB


def dump_outputs(out_dir, frame):
    """Write the frame of the last timed step (RGBA8, un-premultiplied) as float32 `frame.npy`, shape (rows, width, 4), and
    the frame rows it holds as float64 `frame_rows.npy`. A frame larger than DUMP_BYTES is sampled by rows chosen with a
    fixed seed, so two builds run with the same arguments can be compared pixel for pixel."""
    os.makedirs(out_dir, exist_ok=True)
    h, w = frame.shape[:2]
    n = max(1, min(h, DUMP_BYTES // (w * 4 * 4)))
    rows = np.arange(h) if n == h else np.sort(np.random.default_rng(0).choice(h, n, replace=False))
    np.save(os.path.join(out_dir, "frame.npy"), frame[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_rows.npy"), rows.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the single JSON line (no NCCL version banner)
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return rank, world, local, dist
    return rank, world, local, None


from vello_b200.stripes import stripe_for  # noqa: E402  (bin-row stripe of a rank)


def run_cpu_arm(args, packed, as_reference):
    """Time the oracle (restated reference CPU shaders + fine) on the host cores."""
    from oracle.vbo import Oracle
    from vello_b200.encoding import BLACK
    cores = os.cpu_count() or 1
    o = Oracle(threads=cores)
    # one full frame is ~3-5 s of CPU work on 8 cores, so the reference arm runs at most one warm-up frame; it times
    # exactly --steps frames (the cpu_baseline beside the GPU figure times one)
    steps = args.steps if as_reference else 1
    warm = min(args.warmup, 1) if as_reference else 0
    times, serial, fine = [], [], []
    w, h = args.size, args.height or args.size
    frame = None
    for i in range(warm + steps):
        t = time.perf_counter()
        o.bind(packed, w, h, BLACK.premul_rgba8_u32(), args.aa)
        o.run("pathtag", "path_tiling")  # one host thread, like the reference's CPU shaders (RendererOptions::use_cpu)
        t1 = time.perf_counter()
        frame = o.run("fine", "fine")    # the reference has no CPU fine; ours runs one thread per tile row, all cores
        t2 = time.perf_counter()
        if i >= warm:
            times.append(t2 - t)
            serial.append(t1 - t)
            fine.append(t2 - t1)
    fps = len(times) / sum(times)
    fine_threads = min(cores, 1024, (h + 15) // 16)
    return fps, dict(value=fps, unit="frames/s", cores=cores, kind="port",
                     sample=f"{len(times)} full frame(s) of the workload; pathtag..path_tiling on ONE thread as the reference's CPU shaders run "
                            f"({1000 * sum(serial) / len(serial):.0f} ms/frame), fine on {fine_threads} threads ({1000 * sum(fine) / len(fine):.0f} ms/frame)"), \
        1000.0 * sum(times) / len(times), len(times), frame


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries print to fd 1 behind Python's back (NCCL's version banner, for one). Everything that is not the JSON
    # line is sent to stderr: fd 1 is re-pointed at fd 2 for the run and the line is written to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--paths", type=int, default=WORKLOAD["n_paths"])
    ap.add_argument("--size", type=int, default=WORKLOAD["size"])
    ap.add_argument("--seed", type=int, default=WORKLOAD["seed"])
    ap.add_argument("--aa", type=int, default=WORKLOAD["aa"])
    ap.add_argument("--scene", default="paris", choices=["paris", "tiger", "beziers"], help="paris = the headline workload")
    ap.add_argument("--height", type=int, default=0, help="frame height (default: --size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-exchange", action="store_true", help="N > 1: every rank flattens the whole scene (round-1 behaviour)")
    ap.add_argument("--profile-only", action="store_true", help="just run warmup+steps resident frames (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if not args.profile_only else args.warmup

    H = args.height or args.size
    wl = {"paris": f"paris-like-{args.paths // 1000}k", "tiger": "Ghostscript tiger", "beziers": f"beziers-{args.paths // 1000}k+clips"}[args.scene]
    config = {"workload": f"{wl} {args.size}x{H} " + ["Area", "MSAA8", "MSAA16"][args.aa],
              "n_paths": args.paths, "seed": args.seed, "parallelism": f"tile-row stripes x{args.gpus}",
              "l2": "flushed between steps (256 MiB write) outside the per-step CUDA-event pairs"}

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        packed, _ = build_scene(args)
        fps, cb, ms, n, frame = run_cpu_arm(args, packed, True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, frame)
        emit({"impl": "reference", "metric": "frames/sec paris-30k@4K", "value": fps, "unit": "frames/s",
                          "n_gpus": args.gpus, "steps": n, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": cb, "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0})
        return

    rank, world, local, dist = dist_setup(args.gpus)
    import torch
    from vello_b200.config import RenderParams
    from vello_b200.encoding import BLACK
    from vello_b200.renderer import Renderer, RendererOptions, FrameStats, _Layout, _Params
    from vello_b200.stripes import even_tile_bounds, rebalance

    packed, gen_s = build_scene(args)
    params = RenderParams(BLACK, args.size, H, args.aa)
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    r = Renderer(RendererOptions(device=local))
    r.upload(packed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(r.stream, device=dev)
    vp = C.c_void_p

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allgather_floats(v):
        if dist is None:
            return [list(v)]
        t = torch.tensor(list(v), dtype=torch.float64, device=dev)
        outs = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(outs, t)
        return [o.tolist() for o in outs]

    # ---- the frame buffer. One GPU: a device buffer. N GPUs: the frame lives on rank 0 (allocated by the library, exported
    # through CUDA IPC) and every rank's `fine` stores its stripe STRAIGHT INTO IT over NVLink peer mapping -- no gather pass.
    frame_bytes = args.size * H * 4
    frame_ptr = vp()
    if rank == 0:
        assert r.lib.vb_frame_alloc(r.handle, frame_bytes, C.byref(frame_ptr)) == 0
    if world > 1:
        handle = C.create_string_buffer(64)
        if rank == 0:
            assert r.lib.vb_ipc_export(r.handle, frame_ptr, handle) == 0
        ht = torch.tensor(list(handle.raw), dtype=torch.uint8, device=dev)
        dist.broadcast(ht, src=0)
        ok = 1.0
        if rank != 0:
            hb = C.create_string_buffer(bytes(ht.cpu().tolist()), 64)
            rc = r.lib.vb_ipc_open(r.handle, hb, C.byref(frame_ptr))
            if rc != 0:
                print(f"rank {rank}: vb_ipc_open failed ({r.lib.vb_last_error(r.handle).decode()}): stripes stay on their GPUs", file=sys.stderr)
                ok = 0.0
        okt = torch.tensor([ok], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        p2p_frame = okt.item() > 0.0
    else:
        p2p_frame = True
    frame_base = int(frame_ptr.value or 0)
    if args.dump_outputs and not p2p_frame:
        raise SystemExit("--dump-outputs: the stripes stay on their GPUs (no peer mapping of rank 0's frame), so no rank holds the frame")

    bounds = even_tile_bounds(world, H)

    def my_rows():
        return (bounds[rank], bounds[rank + 1]) if world > 1 else (0, 0)

    def my_out():
        if world > 1 and not p2p_frame:
            return 0  # no peer mapping of rank 0's frame on this box: every rank keeps its stripe (the renderer's own target)
        return frame_base + (bounds[rank] * 16 * args.size * 4 if world > 1 else 0)

    def render_once():
        return r.render_resident(params, my_out(), tile_rows=my_rows())

    # ---- warm-up: size the arenas, then (N > 1) move the stripe boundaries until the ranks take equally long
    st = render_once()
    balance_log = []
    if world > 1:
        for it in range(12):
            for _ in range(2):
                render_once()
            ms = [v[0] for v in allgather_floats([float(r.lib.vb_last_frame_ms(r.handle))])]
            balance_log.append({"bounds": list(bounds), "ms": [round(m, 4) for m in ms]})
            nb = rebalance(bounds, ms)
            if nb == bounds:
                break
            bounds = nb
    # ---- N > 1: shard flatten by tag range and exchange lines / path boxes through peer memory (k_exchange.cu). The frames
    # above (every rank flattening everything) are the `replicated` figure reported beside `value`.
    replicated = None
    exchange_on = world > 1 and not args.no_exchange
    xinfo = None

    def render_collective():
        """One frame on every rank; re-issued on every rank while any rank's arenas overflow (exchanged frames advance an
        epoch on all GPUs together)."""
        nonlocal st
        for attempt in range(10):
            ps_ = _Params(BLACK.premul_rgba8_u32(), args.size, H, args.aa, 0, 0, my_rows()[0], my_rows()[1])
            fs_ = FrameStats()
            rc = r.lib.vb_render_resident(r.handle, C.byref(ps_), vp(my_out()), C.byref(fs_))
            bad = torch.tensor([1.0 if rc != 0 else 0.0], device=dev)
            dist.all_reduce(bad, op=dist.ReduceOp.MAX)
            if bad.item() == 0.0:
                st = fs_
                return attempt
            assert rc in (0, -3), f"rank {rank}: vb_render_resident rc={rc} [{r.lib.vb_last_error(r.handle).decode()}]"
        raise RuntimeError("exchanged frame kept overflowing")

    if exchange_on:
        # the replicated mode's K steps first (same protocol as the main loop below)
        for _ in range(args.warmup):
            render_once()
        barrier()
        evs0 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in evs0:
            flush.fill_(1)
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            a.record(stream)
            r.enqueue(params, my_out(), tile_rows=my_rows())
            b.record(stream)
            assert r.finish().failed == 0
        barrier()
        sm0 = torch.tensor([a.elapsed_time(b) for a, b in evs0], dtype=torch.float64, device=dev)
        dist.all_reduce(sm0, op=dist.ReduceOp.MAX)
        replicated = {"value": args.steps / (float(sm0.sum().item()) / 1000.0), "unit": "frames/s", "ms_per_step": float(sm0.sum().item()) / args.steps,
                      "tile_row_bounds": list(bounds), "note": "every rank flattens the whole scene (culled to its stripe); no exchange"}
        # arenas, CUDA IPC handles all-gathered, peers mapped (any failure on any rank: everybody stays in replicated mode)
        arena, nbytes = vp(), C.c_size_t(0)
        xok = 1.0 if r.lib.vb_exchange_configure(r.handle, rank, world, C.byref(arena), C.byref(nbytes)) == 0 else 0.0
        hb = C.create_string_buffer(64)
        if xok and r.lib.vb_ipc_export(r.handle, arena, hb) != 0:
            xok = 0.0
        mine = torch.tensor(list(hb.raw), dtype=torch.uint8, device=dev)
        allh = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allh, mine)
        okt = torch.tensor([xok], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        peer_ptrs = []
        if okt.item() > 0.0:
            for k in range(world):
                if k == rank:
                    continue
                hk = C.create_string_buffer(bytes(allh[k].cpu().tolist()), 64)
                pk = vp()
                if r.lib.vb_ipc_open(r.handle, hk, C.byref(pk)) != 0 or r.lib.vb_exchange_attach(r.handle, k, pk) != 0:
                    print(f"rank {rank}: could not map the exchange arena of rank {k}: {r.lib.vb_last_error(r.handle).decode()}", file=sys.stderr)
                    xok = 0.0
                    break
                peer_ptrs.append(pk)
            okt = torch.tensor([xok], device=dev)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        exchange_on = okt.item() > 0.0
        if not exchange_on:
            xinfo = {"chosen": "replicated", "why": "exchange arenas could not be set up on this box"}
    if exchange_on:

        def set_bounds():
            arr = (C.c_uint32 * (world + 1))(*bounds)
            assert r.lib.vb_exchange_set_bounds(r.handle, arr) == 0

        set_bounds()
        assert r.lib.vb_exchange_enable(r.handle, 1) == 0
        barrier()
        retries = render_collective()
        xbal = []
        for it in range(12):  # re-balance: the replicated flatten is gone, the stripes weigh differently now
            for _ in range(2):
                render_collective()
            ms = [v[0] for v in allgather_floats([float(r.lib.vb_last_frame_ms(r.handle))])]
            xbal.append({"bounds": list(bounds), "ms": [round(m, 4) for m in ms]})
            nb = rebalance(bounds, ms)
            if nb == bounds:
                break
            bounds = nb
            set_bounds()
        xinfo = {"arena_bytes": int(nbytes.value), "first_frame_reissues": retries, "balancing": xbal,
                 "how": "rank k flattens partitions [P*k/N, P*(k+1)/N) of the tag stream; lines are routed by the stripes they touch into an "
                        "outbox in peer-mapped memory and pulled by their owners, partial path boxes are min/max-combined; the ranks "
                        "synchronise through epoch flags in each other's arenas (no host, no NCCL on the data path)"}

        # which mode is faster depends on N and on the scene (the exchange moves every line once more; it pays when the
        # replicated flatten is a large part of a rank's frame: many GPUs, curve-heavy scenes): calibrate, keep the better one
        cal = []
        for _ in range(8):
            flush.fill_(1)
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            render_collective()
            cal.append(float(r.lib.vb_last_frame_ms(r.handle)))
        tcal = torch.tensor([sum(cal[2:]) / len(cal[2:])], dtype=torch.float64, device=dev)
        dist.all_reduce(tcal, op=dist.ReduceOp.MAX)
        xinfo["calibration_ms"] = float(tcal.item())
        xinfo["replicated_ms"] = replicated["ms_per_step"]
        if float(tcal.item()) > replicated["ms_per_step"]:
            exchange_on = False
            assert r.lib.vb_exchange_enable(r.handle, 0) == 0
            bounds = list(replicated["tile_row_bounds"])
            xinfo["chosen"] = "replicated"
        else:
            xinfo["chosen"] = "exchange"

            def render_once():  # noqa: F811  (from here on every frame is an exchanged one)
                render_collective()
                return st

    for _ in range(args.warmup):
        st = render_once()
    if args.profile_only:
        for _ in range(args.steps):
            render_once()
        return

    # ---- resident-scene throughput ("value"): exactly K steps, CUDA events per step on the renderer's stream, L2 flushed
    # between steps; a step of the N-GPU job lasts as long as its slowest rank, so the per-step times are max-reduced over ranks
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    t_wall = time.perf_counter()
    for a, b in evs:
        flush.fill_(1)          # L2 flush on the default stream ...
        torch.cuda.synchronize()  # ... finished before the step starts
        if dist is not None:
            dist.barrier()      # all ranks start the frame together (one frame = all its stripes)
            torch.cuda.synchronize()
        a.record(stream)
        r.enqueue(params, my_out(), tile_rows=my_rows())
        b.record(stream)
        s = r.finish()
        assert s.failed == 0
        launches += int(s.kernel_launches)
    barrier()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # read back now: the sections below render into the same frame
        last = np.zeros((H, args.size, 4), dtype=np.uint8)
        assert r.lib.vb_copy_to_host(r.handle, vp(frame_base), vp(last.ctypes.data), C.c_size_t(last.nbytes)) == 0
        dump_outputs(args.dump_outputs, last)
        del last
    step_ms = torch.tensor([a.elapsed_time(b) for a, b in evs], dtype=torch.float64, device=dev)
    my_total = float(step_ms.sum().item())
    if dist is not None:
        dist.all_reduce(step_ms, op=dist.ReduceOp.MAX)
    total_ms = float(step_ms.sum().item())
    fps = args.steps / (total_ms / 1000.0)
    rank_totals = [v[0] for v in allgather_floats([my_total])]

    # ---- the same K steps with the stripes LEFT ON THEIR GPUS (every rank paints into its own buffer, no NVLink traffic): at
    # 16384^2 the assembly of 1 GiB per frame on one GPU is bound by that GPU's NVLink ingest (~0.8 TB/s), SURVEY.md 8e asks
    # for both figures
    distributed = None
    if world > 1:
        for _ in range(3):
            r.render_resident(params, 0, tile_rows=my_rows())
        barrier()
        evs2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in evs2:
            flush.fill_(1)
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            a.record(stream)
            r.enqueue(params, 0, tile_rows=my_rows())
            b.record(stream)
            assert r.finish().failed == 0
        barrier()
        sm2 = torch.tensor([a.elapsed_time(b) for a, b in evs2], dtype=torch.float64, device=dev)
        dist.all_reduce(sm2, op=dist.ReduceOp.MAX)
        distributed = {"value": args.steps / (float(sm2.sum().item()) / 1000.0), "unit": "frames/s",
                       "ms_per_step": float(sm2.sum().item()) / args.steps, "note": "stripes left in each GPU's own memory"}

    # ---- the assembled frame: rank 0 renders the whole frame alone and compares (stripes over NVLink == one GPU)
    stripes_parity = None
    if world > 1 and p2p_frame:
        barrier()
        if rank == 0:
            asm = np.zeros((H, args.size, 4), dtype=np.uint8)
            assert r.lib.vb_copy_to_host(r.handle, vp(frame_base), vp(asm.ctypes.data), C.c_size_t(asm.nbytes)) == 0
            if exchange_on:
                assert r.lib.vb_exchange_enable(r.handle, 0) == 0  # a frame of rank 0 alone: nobody to exchange with
            r.render_resident(params, 0)
            solo = r.download_target(params)
            if exchange_on:
                assert r.lib.vb_exchange_enable(r.handle, 1) == 0
            stripes_parity = {"assembled_over_nvlink_equals_single_gpu": bool(np.array_equal(asm, solo)),
                              "differing_pixels": int((asm != solo).any(axis=2).sum())}
            del asm, solo
        barrier()

    # ---- end-to-end through the C ABI with pinned host buffers ("e2e") ---------------------------
    h0, h1 = r.stripe_rows(params, (0, 0), my_rows())
    scene_h = torch.from_numpy(np.ascontiguousarray(packed.scene)).pin_memory()
    ramps_h = torch.from_numpy(np.ascontiguousarray(packed.ramps.reshape(-1))).pin_memory() if packed.ramps.size else None
    atlas_np = np.ascontiguousarray(packed.atlas)
    outs = tuple(torch.empty((max(h1 - h0, 1), args.size, 4), dtype=torch.uint8).pin_memory() for _ in range(3))
    lay = _Layout(*[int(v) for v in packed.layout.as_array()])
    tr = my_rows()
    ps = _Params(BLACK.premul_rgba8_u32(), args.size, H, args.aa, 0, 0, tr[0], tr[1])
    fs = FrameStats()

    def e2e_args(o):
        return (r.handle, scene_h.data_ptr(), scene_h.numel() * 4, C.byref(lay), ramps_h.data_ptr() if ramps_h is not None else None, 512,
                packed.ramps.shape[0], atlas_np.ctypes.data, atlas_np.shape[1], atlas_np.shape[0], C.byref(ps), o.data_ptr())

    def e2e_sync_step():  # one blocking call per frame: upload + render + read-back
        rc = r.lib.vb_render(*e2e_args(outs[0]), 0, C.byref(fs))
        assert rc == 0 and fs.failed == 0

    def e2e_stream(n):  # streaming form: upload(k+1) | raster(k) | read-back(k-1) overlap, three host buffers
        for k in range(n):
            rc = r.lib.vb_render_begin(*e2e_args(outs[k % 3]), C.byref(fs))
            assert rc == 0 and fs.failed == 0
        assert r.lib.vb_readback_wait(r.handle) == 0  # every frame's pixels are in host memory when the clock stops

    e2e_steps = max(6, args.steps // 2)
    e2e_fps_by_mode = {}
    for mode in ("sync", "stream"):
        for _ in range(3):
            e2e_sync_step() if mode == "sync" else e2e_stream(3)
        barrier()
        t0 = time.perf_counter()
        if mode == "sync":
            for _ in range(e2e_steps):
                e2e_sync_step()  # vb_render synchronises internally: host wall clock == device completion
        else:
            e2e_stream(e2e_steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_fps_by_mode[mode] = e2e_steps / float(t.item())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "streamed frames differ"
    e2e_fps = e2e_fps_by_mode["stream"]
    h2d = int(packed.scene.nbytes + packed.ramps.nbytes + packed.atlas.nbytes)
    d2h = int((h1 - h0) * args.size * 4 + 32)

    # ---- per-stage CUDA events of this rank's stripe (the same renderer with timing switched on: plain launches, an event
    # between stages; at N > 1 these are collective frames like all the others, so `flatten` includes the exchange and the wait
    # for the slowest peer)
    assert r.lib.vb_set_timing(r.handle, 1) == 0
    render_once()
    stage_ms = {}
    n_t = 10
    for _ in range(n_t):
        flush.fill_(1)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()
        sd = render_once().as_dict()
        for k, v in sd["stage_ms"].items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v / n_t
    assert r.lib.vb_set_timing(r.handle, 0) == 0
    ptcl_words, seg_refs, fill_cmds = r.fine_traffic()  # what the interpreter reads, from each tile's occlusion start
    r.set_occlusion_cull(False)
    full_words, full_segs, full_fills = r.fine_traffic()  # the whole command lists, as the reference executes them
    r.set_occlusion_cull(True)
    bump = {k: int(getattr(st, k)) for k in ("lines", "tile", "seg_counts", "segments", "ptcl", "binning")}
    stage_by_rank = None
    if dist is not None:
        names = list(stage_ms.keys())
        allv = allgather_floats([stage_ms[k] for k in names])
        stage_by_rank = [{k: round(v, 4) for k, v in zip(names, row)} for row in allv]
    if rank != 0:
        if world > 1:
            r.lib.vb_ipc_close(r.handle, vp(frame_base))
        r.close()
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (fine) and the per-stage table, from algorithmic bytes (SURVEY.md 8d) ----------
    peak, peak_src = measured_peaks()
    px = (h1 - h0) * args.size
    L = packed.layout
    n_tags = int(L.path_data_base - L.path_tag_base) * 4
    n_tag_words = n_tags // 4
    n_paths, n_draw, n_clips = int(L.n_paths), int(L.n_draw_objects), int(L.n_clips)
    points_bytes = int(L.draw_tag_base - L.path_data_base) * 4
    NL, Nx, Ta, W = bump["lines"], bump["seg_counts"], bump["tile"], ptcl_words
    alg = {  # minimum traffic, each datum once
        "pathtag": n_tags + 20 * n_tag_words,
        "flatten": n_tags + 20 * n_tag_words + points_bytes + 24 * NL,
        "draw": 4 * n_draw + 16 * n_draw + 24 * n_paths,
        "clip": 8 * n_clips + 16 * n_clips,
        "binning": 16 * n_draw + 4 * bump["binning"],
        "tile_alloc": 32 * n_draw + 8 * Ta,
        "path_count": 24 * NL + 8 * Nx,
        "backdrop": 16 * Ta,
        "coarse": 8 * Ta + 4 * (full_words if world == 1 else W),
        "path_tiling": 8 * Nx + 24 * Nx + 24 * Nx,
        "fine": 4 * px + 4 * ptcl_words + 24 * seg_refs,
    }
    stages = {k: {"bytes": int(alg[k]), "ms": round(stage_ms[k], 4), "gbs": round(alg[k] / max(stage_ms[k], 1e-9) / 1e6, 1),
                  "frac_of_hbm": round(alg[k] / max(stage_ms[k], 1e-9) / 1e6 / peak, 4)} for k in alg if k in stage_ms}
    scans = {"pathtag_words_per_s": n_tag_words / (stage_ms["pathtag"] / 1e3), "pathtag_tags_per_s": n_tags / (stage_ms["pathtag"] / 1e3),
             "draw_objs_per_s": n_draw / (stage_ms["draw"] / 1e3),
             "pathtag_frac_of_hbm": stages["pathtag"]["frac_of_hbm"], "draw_frac_of_hbm": stages["draw"]["frac_of_hbm"],
             "note": "single-pass decoupled look-back scans; bytes = tags in + 20 B monoid per tag word out (pathtag), "
                     "draw tag + monoid + bbox per object (draw)"}
    alg_bytes = alg["fine"]
    fine_s = stage_ms["fine"] / 1000.0
    achieved = alg_bytes / fine_s / 1e9
    roofline = {"kernel": f"k_fine<{args.aa}>", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes": alg_bytes, "bytes_breakdown": {"pixels": 4 * px, "ptcl": 4 * ptcl_words, "segments": 24 * seg_refs},
                "fine_ms": stage_ms["fine"], "fill_cmds_executed": fill_cmds,
                "whole_list": {"bytes": 4 * px + 4 * full_words + 24 * full_segs, "fill_cmds": full_fills},
                "note": "bytes = pixels + the PTCL words and segments fine reads from each tile's occlusion start (last opaque "
                "full-tile cover, noted by coarse); whole_list = the same count over the complete lists the reference executes. "
                "MSAA16 fine is issue / shared-memory-atomic bound, not HBM bound (SURVEY.md 8d caveat): see issue_bound"}
    # dram traffic and warp-instruction count of k_fine are ncu measurements: they are quoted only when the capture under
    # profiles/ was made with THIS k_fine.cu at THIS configuration (hash + workload recorded beside the numbers), else null
    try:
        import hashlib
        meta = json.load(open(os.path.join(ROOT, "profiles", "fine_ncu.json")))
        src_hash = hashlib.sha256(open(os.path.join(ROOT, "vello_b200", "csrc", "k_fine.cu"), "rb").read()).hexdigest()[:16]
        if meta.get("k_fine_sha16") == src_hash and meta.get("workload") == config["workload"] and world == 1:
            roofline["traffic"] = meta.get("dram_bytes_per_launch")
            wi = meta.get("warp_instructions")
            if wi and clocks and clocks.get("sm_mhz"):
                issue_peak = 148 * 4 * clocks["sm_mhz"] * 1e6  # warp instructions / s: 4 schedulers per SM, one issue per cycle
                roofline["issue_bound"] = {"warp_instructions": wi, "achieved_per_s": wi / fine_s, "peak_per_s": issue_peak,
                                           "frac": wi / fine_s / issue_peak, "source": meta.get("source")}
    except Exception:
        pass

    cpu_baseline, parity = None, {"checked": False}
    if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only (contract)
        # the CPU arm renders this very frame: keep it and compare the GPU's pixels with it (the oracle is the checker here,
        # after every timed region; it is never on the measured path)
        _, cpu_baseline, _, _, cpu_frame = run_cpu_arm(args, packed, False)
        gpu_frame = np.zeros((H, args.size, 4), dtype=np.uint8)
        if world == 1:
            r.render_resident(params, frame_base)
        assert r.lib.vb_copy_to_host(r.handle, vp(frame_base), vp(gpu_frame.ctypes.data), C.c_size_t(gpu_frame.nbytes)) == 0
        d = np.abs(gpu_frame.astype(np.int16) - cpu_frame.astype(np.int16))
        parity = {"checked": True, "against": "oracle (cpu_baseline frame)", "rows": [0, int(H)], "max_diff": int(d.max()) if d.size else 0,
                  "differing_channel_values": int((d > 0).sum()), "tolerance": 0 if args.aa else 1}
        try:  # BASELINE.md 4: the named CPU baseline is sparse_strips/vello_cpu; it needs a Rust toolchain
            has_cargo = subprocess.run(["cargo", "--version"], capture_output=True).returncode == 0
        except Exception:
            has_cargo = False
        cpu_baseline["vello_cpu"] = ("cargo present but the reference tree is not on this box" if has_cargo
                                     else "not buildable: no cargo / rustc on this box (probed), crates not vendored")
    if stripes_parity is not None:
        parity["stripes"] = stripes_parity

    config["parallelism"] = (f"tile-row stripes x{world}, cost-balanced, fine stores into rank 0's frame over NVLink (CUDA IPC)"
                             if world > 1 else "1 GPU")
    line = {"metric": "frames/sec paris-30k@4K", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "vb_render_begin x steps + vb_readback_wait (host scene in, host pixels out, every frame; three frames in flight)",
                    "blocking_vb_render_value": e2e_fps_by_mode["sync"]},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
            "stage_ms": stage_ms, "stages": stages, "scans": scans, "bump": bump,
            "scene_bytes": int(packed.scene.nbytes), "wall_s_timed_region": wall, "scene_build_s": gen_s}
    if world > 1:
        slow = int(np.argmax(rank_totals))
        line["multi_gpu"] = {"flatten": "sharded by tag range, peer-memory exchange" if exchange_on else "replicated", "exchange": xinfo,
                             "replicated": replicated,
                             "tile_row_bounds": list(bounds), "rank_ms_per_step": [round(v / args.steps, 4) for v in rank_totals],
                             "slowest_rank": slow, "stage_ms_by_rank": stage_by_rank, "balancing": balance_log,
                             "frame": "assembled on rank 0 by peer stores from every rank's fine kernel", "distributed": distributed}
    emit(line)
    if world > 1:
        dist.barrier()
    r.lib.vb_frame_free(r.handle, vp(frame_base))
    r.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
