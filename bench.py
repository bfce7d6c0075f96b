#!/usr/bin/env python3
"""bench.py — LSD throughput on synthetic 4096x4096 occupancy grids (BASELINE.json configs[2]).

A "step" = one pass of the LSD hot path (remap + Gaussian + gradient, pseudo-ordering, region grow /
rectangle / NFA) over one batch of `--maps-per-gpu` (256) synthetic maps per GPU.  Weak scaling: every
rank owns its own 256 maps (seed 1000 + global index), no data-path collective.
  value : whole-job source Mpixel/s with the maps already resident in HBM (CUDA events, max over ranks)
  e2e   : the same through the C ABI with HOST buffers — H2D of the maps + run + D2H of the segments
          inside the timed region
  roofline : the HBM-bound stencil kernel, algorithmic bytes N + 17n per map over its measured time
  cpu_baseline : the unmodified reference (oracle/_ref, stock glibc) on a bounded sample of the same maps
`--impl reference` times that CPU reference alone (rank 0 only), one map per host thread.
`--dump-outputs DIR` writes rank 0's segment tables of the last timed step as .npy files (see dump_outputs) so that two
builds can be compared output for output: the inputs depend on the arguments only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "lsd_source_mpixel_per_s"
UNIT = "Mpixel/s"


def make_map(size, gidx):
    import synth
    return synth.occupancy_grid(size, size, seed=1000 + gidx)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_throughput(size, n_maps, threads, first_gidx=0):
    """The unmodified reference myLineSegmentDetector (oracle/_ref, stock glibc) on n_maps of the workload,
    one map per host thread (the reference is single-threaded per map; ctypes releases the GIL)."""
    import refbind
    if not refbind.available("glibc"):
        return None
    maps = [make_map(size, first_gidx + i) for i in range(n_maps)]
    counts = [0] * n_maps

    def work(tid):
        for i in range(tid, n_maps, threads):
            counts[i] = refbind.ref_lsd(maps[i], want_maps=False)["n"]

    t0 = time.time()
    th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.time() - t0
    return dict(seconds=dt, mpix_per_s=n_maps * size * size / dt / 1e6, segments=int(sum(counts)), n_maps=n_maps)


DUMP_LIMIT = 64 * 10**6


def split_nonfinite(a):
    """a 2-D array -> (a with its non-finite entries set to 0, one (row, column, code) record per such entry; code 1 = +inf,
    -1 = -inf, 2 = NaN), both finite float64: vertical segments carry k = -inf, b = NaN (structLinesInfo)."""
    bad = ~np.isfinite(a)
    r, c = np.nonzero(bad)
    code = np.where(np.isnan(a[r, c]), 2.0, np.sign(a[r, c]))
    return np.where(bad, 0.0, a), np.stack([r, c, code], axis=1).astype(np.float64)


def dump_outputs(out_dir, got, lines_to_array):
    """Writes what a caller of the timed path receives, as finite float64 .npy files under out_dir: counts (segments per map),
    maps (the indices of the maps whose tables follow), lines (structLinesInfo in oracle column order) and rects (rectangle and
    log-NFA records), the tables of those maps concatenated in map order, with their non-finite entries in lines_nonfinite /
    rects_nonfinite (see split_nonfinite).  Every map when the files fit in DUMP_LIMIT bytes, else a fixed seeded sample of
    the maps."""
    counts = np.asarray(got["counts"], np.int64)
    tables = [(lines_to_array(got["lines"][i]), got["rects"][i]) for i in range(counts.size)]
    map_bytes = np.array([8 * (ln.size + rc.size) + 24 * int((~np.isfinite(ln)).sum() + (~np.isfinite(rc)).sum()) for ln, rc in tables])
    budget = DUMP_LIMIT - 2 * 8 * counts.size - 6 * 128     # counts, maps and the six .npy headers
    order = np.arange(counts.size)
    if map_bytes.sum() > budget:
        order = np.random.default_rng(0).permutation(counts.size)
    maps = np.sort(order[np.cumsum(map_bytes[order]) <= budget])
    lines, lines_nf = split_nonfinite(np.concatenate([np.zeros((0, 10))] + [tables[i][0] for i in maps]))
    rects, rects_nf = split_nonfinite(np.concatenate([np.zeros((0, 13))] + [tables[i][1] for i in maps]))
    out = {"counts": counts.astype(np.float64), "maps": maps.astype(np.float64), "lines": lines, "lines_nonfinite": lines_nf,
           "rects": rects, "rects_nonfinite": rects_nf}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def stencil_traffic(n, size):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE stencil launch (lsdb_stencil2_kernel), from this round's ncu
    capture (profiles/r2_stencil_traffic.json, written by tools/stencil_traffic.py from the .ncu-rep), scaled to this
    launch's source pixels.  None when no capture of this round is on record."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_stencil_traffic.json")))
        return float(t["dram_bytes"]) * (n * size * size) / float(t["source_pixels"])
    except Exception:
        return None


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = min(cores, args.ref_threads or cores)
    k_run, w_run = args.steps, args.warmup   # a step is one map per host thread: ~30 s at 4096^2
    sample = f"{threads} maps of {args.size}x{args.size} per step, one per host thread (of the {args.maps_per_gpu}-map batch)"
    for s in range(w_run):
        r = cpu_reference_throughput(args.size, threads, threads)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_glibc.so not built"}))
            return
    t_all, px = 0.0, 0
    for s in range(k_run):
        r = cpu_reference_throughput(args.size, threads, threads, first_gidx=s * threads)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_glibc.so not built"}))
            return
        t_all += r["seconds"]; px += r["n_maps"] * args.size * args.size
    v = px / t_all / 1e6
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": k_run, "warmup": w_run,
        "ms_per_step": t_all / k_run * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": f"synthetic {args.size}x{args.size} occupancy grids (BASELINE configs[2])",
                                        "maps_per_step": threads},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def run_giant(args, rank, world, local):
    """BASELINE configs[4]: ONE synthetic map (seed 5000) tiled over the ranks — row bands of the stencil stage, NCCL exchange
    of the bands, max-all-reduce of maxGrad, ordering + the sequential seed loop on rank 0 (giant.lsd_tiled).  A step = the
    whole map once; value = source Mpixel/s with the map resident, e2e adds the H2D of the map on every rank and the D2H of
    the tables.  The result of the last step is compared with the CPU oracle on rank 0 (unless --parity-maps 0)."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from __graft_entry__ import load_package
    lsdb = load_package()
    from lsdb200 import giant
    import synth
    size = args.giant_size
    host = torch.from_numpy(synth.occupancy_grid(size, size, seed=5000)).pin_memory()
    m = host.numpy()
    torch.cuda.set_stream(torch.cuda.Stream())
    ctx = lsdb.Context(local, torch.cuda.current_stream().cuda_stream)
    for _ in range(max(args.warmup, 1)):
        out, info = giant.lsd_tiled(ctx, m, rank, world)
    sampler = ClockSampler(local); sampler.start()
    ts, infos = [], []
    for _ in range(args.steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        out, info = giant.lsd_tiled(ctx, m, rank, world)
        torch.cuda.synchronize()
        ts.append((time.time() - t0) * 1e3); infos.append(info)
    clocks = sampler.stop()
    t = torch.tensor([float(np.mean([i["total_ms"] for i in infos])), float(np.mean(ts)), float(np.mean([i["stencil_ms"] for i in infos]))],
                     dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_e2e, ms_stencil = (float(x) for x in t.tolist())
    sent = torch.tensor([float(infos[-1]["bytes_sent_by_this_rank"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(sent)
    if rank == 0:
        parity = None
        if args.parity_maps > 0:
            import oraclebind
            o = oraclebind.lsd(m, want_maps=False, want_line_im=False, max_lines=65536)
            parity = bool(int(out["counts"][0]) == o["n"] and np.array_equal(out["rects"][0], o["rects"], equal_nan=True))
            if not parity:
                raise SystemExit("bench.py: PARITY FAILURE on the tiled map")
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        W = int(size * 0.3); band_px = (infos[-1]["band_rows"][1] - infos[-1]["band_rows"][0]) * W
        alg = size * size * (infos[-1]["band_rows"][1] - infos[-1]["band_rows"][0]) / infos[-1]["scaled_rows"] + 17 * band_px
        line = {"metric": METRIC, "value": size * size / (ms_step * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 1), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "parity_checked_maps": 1 if parity else 0,
                "config": {"workload": f"ONE synthetic {size}x{size} occupancy grid tiled over {world} GPU(s) (BASELINE configs[4])",
                           "partition": "row bands of whole tile rows (32 scaled rows); whole source on every GPU, no halo exchange",
                           "l2": f"the map's planes ({36.25 * W * W / 1e6:.0f} MB) exceed the 126 MB L2"},
                "segments_per_step": int(out["counts"][0]),
                "stage_ms": {"stencil_band_max_over_ranks": ms_stencil, "exchange": infos[-1]["exchange_ms"], "regions_rank0": infos[-1]["regions_ms"]},
                "exchange": {"collectives": "all_reduce(MAX, 1 x f64) + one broadcast per band and plane (in-place all-gather)",
                             "bytes_sent_all_ranks": float(sent.item()), "bytes_per_scaled_row": infos[-1]["bytes_per_scaled_row"]},
                "e2e": {"value": size * size / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": size * size,
                        "d2h_bytes_per_step": int(out["counts"][0]) * 13 * 8 + 128,
                        "how": "Batch create + lsdb_batch_upload of the whole map from pinned host memory on every rank + tiled run + download on rank 0"},
                "gpu_launches": 6 * args.steps,   # stencil tiles + its deferred pixels, ordering x3, regions (rank 0)
                "clocks": clocks,
                "roofline": {"kernel": "lsdb_stencil2_kernel on this rank's band", "bound": "hbm", "achieved": alg / (ms_stencil * 1e-3) / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": alg / (ms_stencil * 1e-3) / 1e9 / peak, "traffic": None,
                             "algorithmic_bytes_per_launch": alg, "kernel_ms": ms_stencil},
                "note": "the seed loop is one sequential chain over the map: the region stage runs on rank 0 and does not shrink with the GPU count"}
        if not args.no_cpu_baseline and args.parity_maps > 0:
            t0 = time.time(); oraclebind.lsd(m, want_maps=False, want_line_im=False, max_lines=65536); dt1 = time.time() - t0
            line["cpu_baseline"] = {"value": size * size / dt1 / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"the whole map once, oracle C port, {dt1:.1f} s"}
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8, help="timed steps of the resident loop (the headline value) and of --impl reference; "
                    "the end-to-end leg runs a multiple of the batches in flight, at least four per batch")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--maps-per-gpu", type=int, default=256)
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--cpu-sample-maps", type=int, default=0, help="maps for the cpu_baseline leg (0 = one per core, max 8)")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inflight", type=int, default=0, help="resident batches that alternate on their own streams (0 = five 256-map batches' worth of maps, 5..12)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank owns --maps-per-gpu maps; strong: the global batch is --maps-per-gpu maps, split over the ranks "
                         "(BASELINE configs[2] as written: batch 256 sharded over 1/2/4/8 GPUs)")
    ap.add_argument("--e2e-line-images", default="auto", choices=["auto", "on", "off"],
                    help="the end-to-end leg also produces every map's lineIm (rasterised on the device, copied to pinned host memory) — "
                         "the reference's call returns it (LSD/myLSD.cpp:296-355); auto = when the host has the memory for the buffers")
    ap.add_argument("--workload", default="batch", choices=["batch", "giant"],
                    help="batch: BASELINE configs[2] (the headline); giant: ONE --giant-size^2 map tiled over the ranks (configs[4])")
    ap.add_argument("--giant-size", type=int, default=16384)
    ap.add_argument("--parity-maps", type=int, default=8, help="maps of the timed batch whose segment tables are checked against the CPU oracle (rank 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's segment tables of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "batch"):
        ap.error("--dump-outputs needs --impl b200 --workload batch")

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "giant":
        run_giant(args, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from __graft_entry__ import load_package
    lsdb = load_package()
    from lsdb200 import shard
    # two explicit streams: their handles are what the library launches on.  Two resident batches (A, B) of the same
    # maps alternate, step by step: while the last, slow maps of one step finish, the next step's maps already occupy the
    # SMs they left idle — the steady state of a caller that keeps the device fed.
    size = args.size
    if args.scaling == "strong":
        global_n = args.maps_per_gpu                          # strong scaling: ONE batch of --maps-per-gpu maps, split over the ranks
        first, n = shard.shard_range(global_n, rank, world)
        if n <= 0:
            raise SystemExit("bench.py: more ranks than maps")
    else:
        n = args.maps_per_gpu
        global_n = world * n
        first, cnt = shard.shard_range(global_n, rank, world)   # weak scaling: every rank owns n maps of the global batch
        assert cnt == n
    # batches in flight: enough to keep ~1280 maps on the device (what five 256-map batches are) when a rank's share is smaller
    # (strong scaling), at most 12; the region stage's rate depends on how many maps are resident, not on how they are batched
    NB = args.inflight if args.inflight > 0 else max(5, min(12, -(-1280 // n)))
    team_note = "library default"
    streams = [torch.cuda.Stream() for _ in range(NB)]
    torch.cuda.set_stream(streams[0])
    stream = streams[0]
    ctxs = [lsdb.Context(local, st.cuda_stream) for st in streams]
    ctx = ctxs[0]
    # Team size of the region stage.  The library picks it as if a batch were alone on the device (4 warps per map at 256 maps,
    # 8 below ~150).  With NB batches in flight the device is full of maps, the stage is bound by instruction supply (DESIGN.md
    # §4.3) and smaller teams do less speculative work per map: measured 250.8 / 189.8 / 207.6 / 216.6 ms per 256-map step with
    # 1 / 2 / 3 / 4 warps per map (1 184 two-warp teams fit on 148 SMs).
    tw = 0
    if "LSDB_GROW_WARPS" not in os.environ:
        tw = 2 if NB * n >= 1184 else (4 if n < 256 and NB * n >= 256 else 0)
        if tw:
            for c_ in ctxs:
                c_.set_team_warps(tw)
            team_note = f"{tw} warps per map (lsdb_set_team_warps: the batches in flight fill the device)"
    host = torch.empty((n, size, size), dtype=torch.uint8).pin_memory()
    hnp = host.numpy()
    for i in range(n):
        hnp[i] = make_map(size, first + i)
    ptrs = [int(hnp[i].ctypes.data) for i in range(n)]
    batches = [lsdb.Batch(c, [(size, size)] * n) for c in ctxs]
    batch = batches[0]
    W = batch.scaled(0)[0]; npx = W * batch.scaled(0)[1]
    src_px = n * size * size

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident: inputs already in HBM
    for bt in batches:
        bt.upload(ptrs)
    for k in range(max(args.warmup, 3, NB)):
        batches[k % NB].run()
    for bt in batches:
        bt.sync()
    sampler = ClockSampler(local); sampler.start()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(NB)]
    e0.record(streams[0])
    for k in range(1, NB):
        streams[k].wait_event(e0)
    for k in range(args.steps):
        batches[k % NB].run()
    for k in range(NB):
        ends[k].record(streams[k])
    barrier()
    ms_total = max(e0.elapsed_time(ev) for ev in ends)
    clocks = sampler.stop()
    # ---------------- the bench checks what it times: segment tables of the first maps of the timed batch against the CPU
    # oracle (bit for bit), before anything else touches the batches.  A mismatch fails the bench.
    parity_k = 0
    if rank == 0 and (args.parity_maps > 0 or args.dump_outputs):
        got0 = batches[(args.steps - 1) % NB].download(want_rects=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, got0, lsdb.lines_to_array)
    if rank == 0 and args.parity_maps > 0:
        import oraclebind
        parity_k = min(args.parity_maps, n)
        for i in range(parity_k):
            o = oraclebind.lsd(hnp[i], want_maps=False, want_line_im=False, max_lines=4096)
            ok = int(got0["counts"][i]) == o["n"] and np.array_equal(got0["rects"][i], o["rects"], equal_nan=True) and \
                np.array_equal(lsdb.lines_to_array(got0["lines"][i]), o["lines"], equal_nan=True)
            if not ok:
                raise SystemExit(f"bench.py: PARITY FAILURE on map {i} of the timed batch: {int(got0['counts'][i])} segments vs {o['n']} from the oracle")
    # one step alone (nothing else on the device): per-stage times from the library's own events on its stream
    batch.run(); batch.sync()
    last = batch.stage_ms()
    stats = batch.stats()
    counts = batch.counts()
    launches_per_step = batch.launches()
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    per_rank = [ms_total / args.steps]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [float(x.item()) / args.steps for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    total_px = global_n * size * size
    value = total_px / (ms_step * 1e-3) / 1e6

    # ---------------- end to end through the C ABI with host buffers
    # Every step copies its 256 maps from pinned host memory, runs the pipeline and reads the segment tables back.
    # Two batches on two private streams alternate (one host thread each; ctypes drops the GIL), so the H2D copy of
    # one step overlaps the kernels of the other: the steady state of a caller that streams batches through the library.
    # The copy phases of a worker leave the device less full than the resident loop does: the library's 4-warp teams are the faster
    # ones here (measured, 20 steps: 19.7 Gpixel/s against 18.0 with 2-warp teams) — fresh batches with that team size.
    e2e_team_note = team_note
    if tw == 2:
        for bt in batches:
            bt.close()
        for c_ in ctxs:
            c_.set_team_warps(4)
        batches = [lsdb.Batch(c, [(size, size)] * n) for c in ctxs]
        batch = batches[0]
        e2e_team_note = "4 warps per map (the library's choice for a 256-map batch)"
    workers = list(zip(ctxs, batches))
    e2e_steps = NB * max(4, (args.steps + NB - 1) // NB)  # a multiple of the worker count; four rounds or more, so that the ramp and the tail of the pipeline do not dominate
    nseg_box = [0] * NB
    # lineIm of every map, too (what the reference's call returns besides the table): one pinned output buffer per worker
    want_im = args.e2e_line_images == "on"
    if args.e2e_line_images == "auto":
        try:
            import psutil
            want_im = psutil.virtual_memory().available / max(world, 1) > (NB * n * size * size) * 2 + (16 << 30)   # every rank allocates its own
        except Exception:
            want_im = False
    im_bufs = [torch.empty((n, size, size), dtype=torch.uint8).pin_memory() for _ in range(NB)] if want_im else []
    im_views = [[bf.numpy()[i] for i in range(n)] for bf in im_bufs]

    def e2e_worker(w, k, with_im):
        cw, bw = workers[w]
        for _ in range(k):
            bw.upload(ptrs); bw.run(); out_w = bw.download()
            if with_im:
                bw.line_images(im_views[w])
            nseg_box[w] = int(out_w["counts"].sum())

    def e2e_run(with_im):
        for w in range(NB):
            e2e_worker(w, 1, with_im)                    # warm-up: allocations, first-touch
        barrier()
        t0 = time.time()
        th = [threading.Thread(target=e2e_worker, args=(w, e2e_steps // NB, with_im)) for w in range(NB)]
        [t.start() for t in th]
        [t.join() for t in th]
        torch.cuda.synchronize()
        dt = torch.tensor([time.time() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return total_px / (float(dt.item()) / e2e_steps) / 1e6

    e2e_tables = e2e_run(False)                          # segment tables only (what round 1 reported)
    e2e_value = e2e_run(True) if want_im else e2e_tables  # + the lineIm of every map: everything the reference's call returns
    nseg = nseg_box[0]
    d2h = n * 4 * 32 + nseg * 13 * 8 + (n * size * size if want_im else 0)   # result records + a rectangle record per segment [+ the lineIm planes]
    if want_im and rank == 0:   # the bench checks what it times: the first map's lineIm against the host epilogue
        if not np.array_equal(im_views[0][0], batches[0].line_image(0)):
            raise SystemExit("bench.py: PARITY FAILURE: device lineIm != host epilogue")
    im_bufs = None; im_views = None
    for cw, bw in workers:
        bw.close()

    # the side measurements below run with the big batches released (they allocate batches of their own)
    for c_ in ctxs:
        c_.set_team_warps(0)   # the side measurements below run one batch at a time: the library's own team sizes
    # ---------------- config 1 latency: the reference's own single-map run (data/mapValue.txt, 1377x428), one map per call
    lat = None
    try:
        if rank != 0:
            raise RuntimeError("side measurements run on rank 0 only")
        g = np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))
        m1 = np.ascontiguousarray(g["mapValue/map"])
        b1 = lsdb.Batch(ctx, [(m1.shape[1], m1.shape[0])])
        b1.upload([m1])
        for _ in range(5):
            b1.run()
        b1.sync()
        ts = []
        for _ in range(50):
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record(stream); b1.run(); eb.record(stream); eb.synchronize()
            ts.append(ea.elapsed_time(eb))
        lat = {"workload": "data/mapValue.txt 1377x428 (BASELINE configs[0]), resident input, batch 1", "p50_ms": float(np.median(ts)),
               "p90_ms": float(np.percentile(ts, 90)), "segments": int(b1.counts()[0]), "runs": len(ts)}
        b1.close()
    except Exception as e:  # the fixture is part of the repo; report rather than hide a failure
        lat = {"error": repr(e)}

    # ---------------- association (BASELINE configs[3] shape): 10k scan frames scored against LSD(data/mapValue.txt) in ONE launch
    fa = None
    try:
        if rank != 0:
            raise RuntimeError("side measurements run on rank 0 only")
        import oraclebind
        gf = np.load(os.path.join(ROOT, "tests", "golden", "fa_frames.npz"))
        gmaps = np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))
        mc = ctx.map_cache(gmaps["mapValue/map"], float(gmaps["mapValue/param"][2]))     # createMapCache on the device
        base = [dict(scan_lines=gf[f"f{f}/scan_lines"], pts=gf[f"f{f}/pts"], lidar_pose=gf[f"f{f}/lidar_pose"],
                     last_pose=[-1.0, -1.0, 0.0]) for f in range(int(gf["n_frames"]))]
        reps = 10000 // len(base) + 1
        frames = base * reps                                                             # 10 008 frames (the 12 reference frames of data/Lidar.txt, tiled)
        fm = lsdb.FaMap(ctx, mc, gf["map_lines"])
        hyp = fm.score(frames)                                                           # warm-up + sizes
        t0 = time.time(); hyp = fm.score(frames); torch.cuda.synchronize(); dt_fa_all = time.time() - t0
        k_ms = fm.last_ms()
        # what a caller of the reference gets back: the hypotheses with score < 3 (LSD/myFA.cpp:261-265).  Host buffers in
        # (the frames packed once into the flat arrays of the C ABI), kept hypotheses out: lsdb_fa_score_kept
        packed = fm.pack(frames)
        # ... in pinned host memory, like the maps of the main leg (the C ABI takes any host pointer; pageable costs ~3x here)
        pins = []   # keeps the pinned storage alive

        def _pin(a):
            if not isinstance(a, np.ndarray) or a.size == 0:
                return a
            t_ = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
            pins.append(t_)
            return t_.numpy().view(a.dtype).reshape(a.shape)

        packed = tuple(_pin(a) for a in packed)
        kept_buf = _pin(np.zeros(len(hyp) // 4 + 4096, lsdb.HYP_DTYPE))                  # the caller's (pinned) table for the kept hypotheses
        kept, n_scored = fm.score_kept(packed, out=kept_buf)                             # warm-up: staging buffers
        t0 = time.time(); kept, n_scored = fm.score_kept(packed, out=kept_buf); dt_fa = time.time() - t0
        assert n_scored == len(hyp) and len(kept) == int((hyp["score"] < 3.0).sum())     # the bench checks what it times
        pts_total = sum(len(f["pts"]) for f in frames)
        # CPU: the reference's own NormalizedLineDirection / rotateScanIm / CalcScore, serial, on the 12 distinct frames
        import refbind
        t0 = time.time(); nh = 0
        for f in base:
            if refbind.available("glibc"):
                idx, _ = refbind.ref_fa_scores(f["scan_lines"], gf["map_lines"], f["pts"], mc, f["lidar_pose"], f["last_pose"])
            else:
                idx, _ = oraclebind.fa_scores(f["scan_lines"], gf["map_lines"], f["pts"], mc, f["lidar_pose"], f["last_pose"])
            nh += len(idx)
        dt_cpu = time.time() - t0
        fa = {"workload": f"{len(frames)} scan frames (12 frames of data/Lidar.txt tiled) x 41 map lines, one launch",
              "hypotheses": int(len(hyp)), "scan_points": int(pts_total), "kernel_ms": k_ms,
              "hypotheses_per_s_kernel": len(hyp) / (k_ms * 1e-3), "hypotheses_per_s_e2e": len(hyp) / dt_fa,
              "e2e_how": "lsdb_fa_score_kept: (pinned) host lines / raster samples in, pair filter + scoring + ordered compaction on the device, "
                         "the hypotheses with score < 3 out into the caller's pinned table", "kept_hypotheses": int(len(kept)),
              "hypotheses_per_s_e2e_all_returned": len(hyp) / dt_fa_all,
              "cpu_reference_hypotheses_per_s": nh / dt_cpu, "cpu_kind": "reference serial (1 thread)" if refbind.available("glibc") else "port",
              "l2_note": "mapCache 1377x428 f64 = 4.7 MB gathers are L2-resident"}
        fm.close()
    except Exception as e:
        fa = {"error": repr(e)}

    # ---------------- scan front-end (SURVEY §8f rank 2): 10k lidar frames -> myrdp::FeatureScan on the device, then the
    # device association reduction on its output (lidar beams in, one pose estimate per frame out)
    fs = None
    try:
        if rank != 0:
            raise RuntimeError("side measurements run on rank 0 only")
        import oraclebind
        import refbind
        gl = np.load(os.path.join(ROOT, "tests", "golden", "lidar_frames.npz"))
        mp = gl["map_param"]
        rng_j = np.random.default_rng(2024)
        base_fr = []
        for f in range(int(gl["n_frames"])):
            r_, a_ = gl[f"f{f}/ranges"], gl[f"f{f}/angles"]
            k_ = np.isfinite(r_)
            base_fr.append((r_[k_], a_[k_]))
        frames_l = []
        for i in range(10000):                                                           # seeded jitter of the bundled sweeps (configs[3])
            r_, a_ = base_fr[i % len(base_fr)]
            frames_l.append((r_ * (1.0 + rng_j.normal(0, 0.002, len(r_))), a_))
        ctx.feature_scan(mp[2], mp[3], mp[4], frames_l[:64])                               # warm-up
        info_, lines_, loff_, pts_, poff_ = ctx.feature_scan(mp[2], mp[3], mp[4], frames_l, raw=True)
        t0 = time.time()
        info_, lines_, loff_, pts_, poff_ = ctx.feature_scan(mp[2], mp[3], mp[4], frames_l, raw=True, capacity=(len(lines_), len(pts_)))
        dt_fs = time.time() - t0
        k_ms = ctx.feature_scan_last_ms()
        gf2 = np.load(os.path.join(ROOT, "tests", "golden", "fa_frames.npz"))
        gm2 = np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))
        fm2 = lsdb.FaMap(ctx, ctx.map_cache(gm2["mapValue/map"], float(gm2["mapValue/param"][2])), gf2["map_lines"])
        fm2.scan_estimate(mp[2], mp[3], mp[4], frames_l[:64])
        fm2.scan_estimate(mp[2], mp[3], mp[4], frames_l)                                   # warm-up: staging buffers
        t0 = time.time()
        _, est_ = fm2.scan_estimate(mp[2], mp[3], mp[4], frames_l)                         # sweeps in, one estimate per frame out
        dt_est = time.time() - t0
        fm2.close()
        # LSD on the scan rasters (configs[3]'s throughput workload): FeatureScan rasters -> occupancy convention -> one batch
        nr = 10000                                                                        # configs[3]: 10k rasterised scans
        sw_ = frames_l[:nr]
        inf_ = ctx.feature_scan_info(mp[2], mp[3], mp[4], sw_)
        rb = lsdb.Batch(ctx, [(int(i_["im_cols"]), int(i_["im_rows"])) for i_ in inf_], max_lines=256)
        rb.upload_scan_rasters(mp[2], mp[3], mp[4], sw_); rb.run(); rb.sync()               # warm-up
        t0 = time.time(); rb.run(); rb.sync(); dt_r = time.time() - t0                       # rasters resident
        t0 = time.time()
        rb.upload_scan_rasters(mp[2], mp[3], mp[4], sw_); rb.run(); r_counts = rb.download()["counts"]   # sweeps in, segment tables out
        dt_re = time.time() - t0
        r_stage = rb.stage_ms(); rb.close()
        r_px = float((inf_["im_cols"].astype(np.int64) * inf_["im_rows"]).sum())
        raster_lsd = {"workload": f"{nr} sweeps -> FeatureScan rasters written into the batch on the device -> LSD (BASELINE configs[3])",
                      "mpix": r_px / 1e6, "ms_resident": dt_r * 1e3, "rasters_per_s_resident": nr / dt_r, "mpix_per_s_resident": r_px / dt_r / 1e6,
                      "ms_e2e": dt_re * 1e3, "sweeps_per_s_e2e": nr / dt_re, "segments": int(r_counts.sum()), "stage_ms": r_stage}
        sample = frames_l[:2000]
        t0 = time.time()
        cpu_nl, _ = refbind.ref_feature_scan_many(list(mp), sample) if refbind.available("glibc") else oraclebind.feature_scan_many(list(mp), sample)
        dt_cpu = time.time() - t0
        assert cpu_nl == int(loff_[len(sample)]) or not refbind.available("lsdm")   # same line count as the device on the sample
        fs = {"workload": f"{len(frames_l)} lidar sweeps (87 bundled Lidar.txt frames, seeded 0.2 % range jitter), one call",
              "beams": int(sum(len(r_) for r_, _ in frames_l)), "lines": int(loff_[-1]), "raster_samples": int(poff_[-1]),
              "kernel_ms_both_passes": k_ms, "frames_per_s_kernel": len(frames_l) / (k_ms * 1e-3),
              "frames_per_s_e2e": len(frames_l) / dt_fs,
              "sweeps_to_estimates_per_s_e2e": len(frames_l) / dt_est, "sweeps_to_estimates_how": "lsdb_scan_estimate_frames, host buffers in/out, incl. the Python marshalling of the sweeps",
              "frames_with_match": int((est_["n_kept"] > 0).sum()), "hypotheses_scored": int(est_["n_hyp"].sum()),
              "cpu_frames_per_s": len(sample) / dt_cpu, "cpu_kind": "reference myrdp::FeatureScan, 1 thread" if refbind.available("glibc") else "port",
              "cpu_sample": "first 2000 frames", "raster_lsd": raster_lsd}
    except Exception as e:
        fs = {"error": repr(e)}


    segs = torch.tensor([float(counts.sum())], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(segs)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6.65 TB/s"
        alg_bytes = n * (size * size + 17 * npx)          # SURVEY §8d: read N source bytes, write mag(8)+deg(8)+used(1) per scaled pixel
        achieved = alg_bytes / (last["stencil"] * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "parity_checked_maps": parity_k,
            "ms_per_step_per_rank": {"min": min(per_rank), "median": float(np.median(per_rank)), "max": max(per_rank), "all": per_rank},
            "config": {"workload": f"synthetic {size}x{size} occupancy grids, global batch {global_n} (BASELINE configs[2]), {n} per GPU",
                       "maps_per_gpu": n, "global_batch": global_n, "parallelism": f"map-sharded x{world}, no collective",
                       "l2": f"inputs {n * size * size / 1e9:.1f} GB per GPU >> 126 MB L2, no flush needed",
                       "pipelining": f"{NB} resident batches alternate on {NB} streams (value and e2e alike); stage_ms / roofline are one step alone",
                       "teams": team_note},
            "segments_per_s": float(segs.item()) / (ms_step * 1e-3), "segments_per_step": float(segs.item()),
            "ms_per_map_amortised": ms_step / n,
            "single_map_latency": lat,
            "association": fa,
            "scan_front_end": fs,
            "stage_ms": last,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * size * size, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "line_images": bool(want_im), "tables_only_value": e2e_tables,
                    "how": "lsdb_batch_upload (pinned host -> HBM) + lsdb_batch_run + lsdb_batch_download" + (" + lsdb_batch_line_images (lineIm of every map -> pinned host)" if want_im else "") + " per step; "
                                               f"{NB} batches on {NB} streams alternate so copies overlap kernels", "teams": e2e_team_note},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "roofline": {"kernel": "lsdb_stencil2_kernel (remap+Gaussian+gradient; + lsdb_stencil_deferred_kernel, 0.02 ms)", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch over 256 maps of 4096^2 (profiles/r1z_ncu_full_summary.txt),
                         # scaled to this launch's map count: the extra over the algorithmic bytes is the cos/sin planes of growable
                         # pixels, the u32 state word (instead of the reference's u8 usedMap) and the ban bit plane
                         "traffic": stencil_traffic(n, size),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": last["stencil"],
                         "share_of_step": last["stencil"] / sum(last.values())},
            "grow_stage": {"bound": "latency", "ms": last["grow"], "share_of_step": last["grow"] / sum(last.values()),
                           "seeds_per_s": stats["live_seeds"] / (last["grow"] * 1e-3),
                           "committed_regions_per_s": (stats["accepts"] + stats["rejects"]) / (last["grow"] * 1e-3),
                           "respeculated_frac": stats["respec_evals"] / max(1, stats["live_seeds"]),
                           "grown_px_per_committed_px_note": "grown_px counts speculative work too",
                           "grown_px": stats["grown_px"], "large_evals": stats["grows"] - stats["small"],
                           "sm_cycles_M": {k: round(stats[k] / 1e6) for k in stats if k.startswith("cyc_")}},
        }
        if not args.no_cpu_baseline and world == 1:
            import refbind
            cores = os.cpu_count() or 1
            if refbind.available("glibc"):
                nm = args.cpu_sample_maps or min(cores, 8)
                th = min(cores, nm)
                r = cpu_reference_throughput(size, nm, th)
                line["cpu_baseline"] = {"value": r["mpix_per_s"], "unit": UNIT, "cores": th, "kind": "reference",
                                        "sample": f"{nm} of the {n} maps ({size}x{size}), one per host thread, {r['seconds']:.1f} s",
                                        "segments": r["segments"]}
            else:
                import oraclebind
                t0 = time.time(); o = oraclebind.lsd(hnp[0], want_maps=False, want_line_im=False); dt1 = time.time() - t0
                line["cpu_baseline"] = {"value": size * size / dt1 / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                        "sample": f"1 of the {n} maps, oracle C port, {dt1:.2f} s"}
        print(json.dumps(line))
    for c in ctxs:
        c.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
