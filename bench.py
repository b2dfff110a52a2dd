#!/usr/bin/env python
"""bench.py -- pose-validity checks/s of the art_planner hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

A "step" is one pass of the hot path over one batch of synthetic input: BASELINE.json configs[1] -- a
1 000 000-pose validity batch (torso + 4 feet, yaml robot geometry) on the fBm ("Perlin") 1000x1000 @0.04 m map.
  value  poses/s with the inputs already resident in HBM (artp_check_poses_bits_device + the ordered index list), CUDA
         events around every step, L2 flushed between timed steps, max over ranks; the library in its shipped default
         (per-stage timing off: the three box kernels of a round run side by side).
  roofline  per-stage kernel durations from a SECOND pass of the same steps with artp_set_timing on (CUDA events recorded
         by the library on the launch stream; the stages then run one after the other) + that pass's throughput
         (serial_order_value).
  e2e    the same metric through the host-buffer C-ABI call (artp_check_poses_f32) with HOST buffers from
         artp_host_alloc: H2D of the 28 B/pose states and D2H of the 1 B/pose mask are inside the timed region; the
         56 B/pose double entry point and a two-caller run are reported beside it; the returned mask is compared with
         the device path's.
  N > 1  weak scaling: every rank checks its own 1 M-pose shard of the seeded sample stream against its replica of
         the map and the ranks exchange the bit-packed verdicts with one NCCL all-gather inside the timed region
         (pipelined; the un-pipelined step is reported too); c5 = configs[4] on spatial map shards (strong scaling).
  --impl reference   the reference's own CPU path (oracle/_ref = its compiled ODE when present, else the C port)
         on all host threads, on a bounded sample of the same workload per step.
  --dump-outputs DIR  after the timed steps, what the last timed step returned as DIR/<name>.npy (float32 / float64,
         exact): valid (verdict bytes), valid_bits (bit-packed verdicts, uint32 words), valid_index (ordered indices of the
         valid samples), valid_count; N > 1: all_valid_bits (the all-gathered masks), written by rank 0. --impl
         reference: valid of its sample. The inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

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

MAP_N = 1000
MAP_RES = 0.04
POSES_PER_GPU = 1_000_000
MAP_SEED, POSE_SEED = 2, 3
WORKLOAD = "configs[1]: fBm 1000x1000@0.04m map (amp 0.6 m), 1M-pose validity batch, yaml robot geometry"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.lines, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "10", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(rank: int, n: int, workload: str = "c2", world: int = 1):
    """c2: BASELINE configs[1] (1000x1000 map; rank r takes samples [r*n, (r+1)*n) of the seeded stream).
    c5: BASELINE configs[4] (4000x4000 map; rank r's samples lie in its spatial slab along x, seed 7)."""
    from art_planner_b200 import synth
    if workload == "c5":
        m = synth.make_fbm_map(4000, 4000, MAP_RES, seed=MAP_SEED, amp=0.6, n_walls=96)
        k = np.arange(rank * n, (rank + 1) * n)
        lx, ly = m.length
        slab = lx * 0.999 / world
        x = m.cx - 0.4995 * lx + (rank + synth.hash_uniform(7, 1, k)) * slab
        y = m.cy + (synth.hash_uniform(7, 2, k) - 0.5) * ly * 0.999
        return m, synth.make_terrain_poses(m, n, seed=7, start=rank * n, xy=(x, y))
    m = synth.make_fbm_map(MAP_N, MAP_N, MAP_RES, seed=MAP_SEED, amp=0.6)
    poses = synth.make_terrain_poses(m, n, seed=POSE_SEED, start=rank * n)
    return m, poses


def dump_outputs(path, arrays):
    """--dump-outputs: one <name>.npy per output array; the integer outputs are written as float64 (exact)."""
    os.makedirs(path, exist_ok=True)
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_oracle(params):
    from oracle import orc
    kind = "reference" if orc.available("reference") else "port"
    if kind == "port":
        orc.build("port")
    return orc.Oracle(params, kind), kind


def best_thread_count(o, poses, cores, big_map=False):
    """The compiled reference stops scaling well before all hardware threads on this host (memory-bound ODE worlds):
    pick the thread count with the highest throughput on a short probe, so the baseline is the reference at its best."""
    cands = sorted({c for c in (8, 16, 32, 64, 128, cores) if c <= cores and (not big_map or c <= 16)})
    best, best_rate = cands[0], 0.0
    probe = poses[:60_000]
    for c in cands:
        o.check_poses_mt(poses[:c * 64], c)          # builds the per-thread ODE worlds (one-time per map, untimed)
        t0 = time.perf_counter(); o.check_poses_mt(probe, c); dt = time.perf_counter() - t0
        if len(probe) / dt > best_rate:
            best, best_rate = c, len(probe) / dt
    return best


STAGE_NAMES = ("aabb", "above", "under", "span", "single_plane", "vertex", "plane_hit", "fall_through")
#: the "rough" level of SURVEY 8(d): fBm with more high-frequency energy; poses aligned to the normal over +-12 cells
#: (= the reference's estimateNormals radius at 0.04 m) so that most torso boxes reach the triangle / plane pass
ROUGH_MAP = dict(amp=1.2, wavelength=3.0, persistence=0.7)
ROUGH_POSES = dict(normal_cells=12)


def exit_mix(port, poses):
    """Per-box exit stage of the reference collider (port statistics, no pose-level short-circuit): torso and feet."""
    st, _, _ = port.pose_box_stats(poses)
    t = np.bincount(st[:, 0], minlength=256)
    f = np.bincount(st[:, 1:].ravel(), minlength=256)
    return {"torso": {k: round(float(t[i]) / len(st), 4) for i, k in enumerate(STAGE_NAMES)},
            "feet": {k: round(float(f[i]) / (4 * len(st)), 4) for i, k in enumerate(STAGE_NAMES)},
            "sample": len(st)}


def pose_workload(torch, chk, flush, m, poses, steps, ref, kind, port, n_mt=400_000, n1=20_000):
    """One 1M-pose validity batch on map m, device-resident: per-stage times, queue sizes, exit mix, and the compiled
    reference (single thread + all threads) on a prefix with the mask compared."""
    n = len(poses)
    chk.setMap(m); chk.updateHeightField(); chk.setTiming(True)
    d = torch.from_numpy(poses).cuda()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        chk.isValidBatch(d, out=out)
    torch.cuda.synchronize()
    ks, tot = [], 0.0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(steps):
        flush.fill_(i & 0xFF)
        a.record(); chk.isValidBatch(d, out=out); b.record()
        ks.append(chk.lastStageTimesMs())
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    st = chk.stats()
    got = out.cpu().numpy()
    k = np.mean(np.array(ks), 0)
    ref.set_map(m); port.set_map(m)
    cores = best_thread_count(ref, poses, os.cpu_count() or 1)
    t0 = time.perf_counter(); v1 = ref.check_poses(poses[:n1]); t1 = time.perf_counter() - t0
    ref.check_poses_mt(poses[:cores * 64], cores)
    t0 = time.perf_counter(); vm = ref.check_poses_mt(poses[:n_mt], cores); tm = time.perf_counter() - t0
    _, zv = port.check_poses(poses[:50_000], want_zone=True)
    return {"map": m.desc, "poses": n, "poses_per_s": n * steps / (tot * 1e-3), "ms_per_step": tot / steps,
            "classify_ms": float(k[0]), "torso_queue_ms": float(k[1]), "reach_queue_ms": float(k[2] + k[3]),
            "reach_queue_warp_ms": float(k[2]), "reach_queue_groups_ms": float(k[3]),
            "group_stage_ms": float(k[4]), "pass_ms": float(k.sum()),
            "queued_boxes": st["last_queued_boxes"], "queued_warp_stage": st["last_queued_warp_stage"],
            "queued_reach_stage": st["last_queued_reach_stage"], "queued_reach_groups": st["last_reach_plane_stage"],
            "deferred_boxes": st["last_deferred"],
            "valid_fraction": float(got.mean()), "exit_mix": exit_mix(port, poses[:20_000]),
            "algorithmic_bytes_per_pose": 57.0 + 4.0 * float(zv.mean()),
            "cpu": {"kind": kind, "single_thread_poses_per_s": n1 / t1, "all_threads_poses_per_s": n_mt / tm, "cores": cores,
                    "sample": f"first {n_mt} poses ({cores} threads), first {n1} (1 thread)",
                    "mask_equals_gpu": bool(np.array_equal(got[:n_mt], vm) and np.array_equal(got[:n1], v1))}}


def run_c5(torch, dist, apb, synth, world, rank, local, flush, steps=5):
    """BASELINE configs[4]: the 4000x4000 map in `world` spatial row slabs (strong scaling: 8 M samples in total). Every rank
    uploads only its slab + a 40-row halo (artp_set_map_window: full-map geometry, local tables), checks the samples that
    fall into its slab, and the ranks all-gather the bit masks. N = 1: the whole map on one GPU."""
    import art_planner_b200  # noqa: F401
    N5, total, halo = 4000, 8_000_000, 40
    n_r = total // world
    m = synth.make_fbm_map(N5, N5, MAP_RES, seed=MAP_SEED, amp=0.6, n_walls=96)
    from art_planner_b200 import sharding
    s0, s1, lo, hi = sharding.slab_window(N5, rank, world, halo)
    chk = apb.StateValidityChecker(synth.PARAMS_YAML, device=local)
    chk.setMap(m)
    t0 = time.perf_counter()
    chk.updateHeightField(window=(lo, hi - lo) if world > 1 else None)
    torch.cuda.synchronize()
    set_map_s = time.perf_counter() - t0
    chk.setTiming(True)
    lx, ly = m.length
    k = np.arange(rank * n_r, (rank + 1) * n_r)
    x_hi, x_lo = m.cx + 0.5 * lx - s0 * MAP_RES, m.cx + 0.5 * lx - s1 * MAP_RES        # x range of the slab's rows
    x = x_lo + (0.0005 + 0.999 * synth.hash_uniform(7, 1, k)) * (x_hi - x_lo)
    y = m.cy + (synth.hash_uniform(7, 2, k) - 0.5) * ly * 0.999
    poses = synth.make_terrain_poses(m, n_r, seed=7, start=rank * n_r, xy=(x, y))
    assert (sharding.rank_of_x(poses[:, 0], m.cx, lx, MAP_RES, N5, world) == rank).all()      # every sample is routed here
    d = torch.from_numpy(poses).cuda()
    v = torch.empty(n_r, dtype=torch.uint8, device="cuda")
    words = (n_r + 31) // 32
    bits = torch.empty(words, dtype=torch.int32, device="cuda")
    idx = torch.empty(n_r, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    all_bits = torch.empty(world * words, dtype=torch.int32, device="cuda") if world > 1 else None

    def step():
        chk.isValidBatchBits(d, v, bits)
        chk.compactValidU32(v, base=0, out_idx=idx, out_cnt=cnt)
        if world > 1:
            dist.all_gather_into_tensor(all_bits, bits)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms, stage = 0.0, []
    for i in range(steps):
        flush.fill_(i & 0xFF)
        a.record(); step(); b.record(); torch.cuda.synchronize()
        ms += a.elapsed_time(b)
        stage.append(chk.lastStageTimesMs())
    chk.pollError()                       # ARTP_E_WINDOW here would mean a sample was routed to the wrong shard
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    st = chk.stats()
    out = None
    if rank == 0:
        o, kind = cpu_oracle(synth.PARAMS_YAML)
        o.set_map(m)                      # the oracle always sees the WHOLE map
        sel = np.arange(0, n_r, 50)
        cores = min(os.cpu_count() or 1, 16)
        t0 = time.perf_counter(); ref = o.check_poses_mt(poses[sel], cores); t_cpu = time.perf_counter() - t0
        got = v.cpu().numpy()
        sm = np.mean(np.array(stage), 0)
        out = {"workload": f"configs[4]: fBm 4000x4000@0.04m map, {total} samples in {world} spatial row slab(s) (+{halo}-row halo), strong scaling",
               "poses_per_s": total * steps / (float(t[0]) * 1e-3), "ms_per_step": float(t[0]) / steps, "steps": steps,
               "samples_per_gpu": n_r, "map_rows_on_gpu": hi - lo if world > 1 else N5,
               "set_map_s": set_map_s, "valid_fraction": float(got.mean()),
               "stage_ms_last_round": dict(zip(("classify", "torso_queue", "reach_queue_warp", "reach_queue_groups", "group"), [float(z) for z in sm])),
               "queued_boxes_last_round": st["last_queued_boxes"],
               "exchange": "one NCCL all-gather of the bit masks per step, inside the timed step (not pipelined)" if world > 1 else "none (N = 1)",
               "mask_equals_reference": bool(np.array_equal(got[sel], ref)),
               "cpu": {"kind": kind, "cores": cores, "poses_per_s": len(sel) / t_cpu,
                       "sample": f"every 50th sample of rank 0's shard ({len(sel)} poses) against the whole map"}}
    del chk
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from art_planner_b200 import synth
    sample_n = 200_000
    m, poses = make_inputs(0, sample_n, getattr(args, "workload", "c2"), 1)
    o, kind = cpu_oracle(synth.PARAMS_YAML)
    o.set_map(m)
    cores = best_thread_count(o, poses, os.cpu_count() or 1, m.rows * m.cols > 4_000_000)
    for _ in range(max(args.warmup, 1)):
        o.check_poses_mt(poses[:20000], cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        valid = o.check_poses_mt(poses, cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"valid": valid.astype(np.float32)})
    value = sample_n * args.steps / dt
    sample = (f"first {sample_n} poses of the 1M-pose workload per step, {cores} threads (best of a probe over "
              f"8..{os.cpu_count()} threads), one ODE world per thread")
    print(json.dumps({
        "impl": "reference", "metric": "pose-validity checks/s", "value": value, "unit": "poses/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": sample_n},
        "cpu_baseline": {"value": value, "unit": "poses/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"],
                    help="c2 = BASELINE configs[1] (default, the metric's config); c5 = configs[4], 4000x4000 map, spatial slabs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import art_planner_b200 as apb
    from art_planner_b200 import build, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()

    n = POSES_PER_GPU
    m, poses = make_inputs(rank, n, args.workload, world)
    chk = apb.StateValidityChecker(synth.PARAMS_YAML, device=local)
    chk.setMap(m)
    chk.updateHeightField()
    chk.setTiming(True)

    d_poses = torch.from_numpy(poses).cuda()
    d_valid = torch.empty(n, dtype=torch.uint8, device="cuda")
    # the adapter's batch buffers: pinned host memory from artp_host_alloc (cudaHostAlloc'd pages: PCIe line rate)
    from art_planner_b200 import capi
    hb_poses, hb_poses32, hb_valid = capi.HostBuffer((n, 7), np.float64), capi.HostBuffer((n, 7), np.float32), capi.HostBuffer((n,), np.uint8)
    hb_poses.array[:] = poses
    hb_poses32.array[:] = poses.astype(np.float32)        # the cast Pose3FromSE3 does first, done by the adapter
    h_poses, h_poses32, h_valid = (torch.from_numpy(x.array) for x in (hb_poses, hb_poses32, hb_valid))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    # Every step produces the verdict bytes, their bit-packed form and the ordered list of valid sample indices of this
    # rank's shard (32-bit, global numbering). N > 1: the ranks exchange the bit masks with ONE NCCL all-gather (125 KB
    # per rank and 10^6 samples); a consumer that wants the global index list reads the per-rank segments + counts.
    assert n % 32 == 0
    my_bits = [torch.empty(n // 32, dtype=torch.int32, device="cuda") for _ in range(2)]
    loc_idx = torch.empty(n, dtype=torch.int32, device="cuda")
    loc_cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    all_bits = torch.empty(world * (n // 32), dtype=torch.int32, device="cuda") if world > 1 else None
    side = torch.cuda.Stream() if world > 1 else None
    ev_done = torch.cuda.Event() if world > 1 else None

    from art_planner_b200 import sharding

    def exchange(b, after_event):
        """The verdict exchange of the step that packed my_bits[b]: runs on the side stream, strictly after
        `after_event` (the START event of the timed window it is accounted to), concurrently with that window's checks."""
        with torch.cuda.stream(side):
            side.wait_event(after_event)
            sharding.gather_valid_bits(my_bits[b], world, out=all_bits)     # 125 KB of mask bits per rank on the wire
            ev_done.record(side)

    def step_device(i, start_event):
        """Window i = checks of step i  ||  exchange of step i-1; the window ends when both are done."""
        if world > 1 and i > 0:
            exchange((i - 1) & 1, start_event)
        chk.isValidBatchBits(d_poses, d_valid, my_bits[i & 1])                  # check + pack, one call
        chk.compactValidU32(d_valid, base=rank * n, out_idx=loc_idx, out_cnt=loc_cnt)   # this shard's ordered index list
        if world > 1 and i > 0:
            torch.cuda.current_stream().wait_event(ev_done)

    def step_serial():
        """The same step without pipelining: check -> pack -> local list -> all-gather, one stream."""
        chk.isValidBatchBits(d_poses, d_valid, my_bits[0])
        chk.compactValidU32(d_valid, base=rank * n, out_idx=loc_idx, out_cnt=loc_cnt)
        if world > 1:
            sharding.gather_valid_bits(my_bits[0], world, out=all_bits)

    def step_e2e():      # what INTEGRATION.md's adapter calls: float32 states (exact), pinned host buffers
        chk.isValidHostPtr(h_poses32.data_ptr(), n, h_valid.data_ptr(), f32=True)

    def step_e2e_f64():  # the same through the double entry point (56 B/pose on the wire)
        chk.isValidHostPtr(h_poses.data_ptr(), n, h_valid.data_ptr())

    # clocks / throttle reasons are sampled every 10 ms from before the warm-up to the end of the end-to-end region
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("ARTP_BENCH_NO_SAMPLER"):   # (experiment switch: how much the 10 ms nvidia-smi polling costs)
        sampler.start()
    warm_ev = torch.cuda.Event()
    for i in range(max(args.warmup, 3)):
        warm_ev.record()
        step_device(i, warm_ev)
    if world > 1:
        warm_ev.record()
        exchange((max(args.warmup, 3) - 1) & 1, warm_ev)
    step_e2e()
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs --------------------------------------------------
    # The library's per-stage event timing is OFF here: that is the shipped default, in which the three box kernels of a
    # round run side by side on internal streams. The per-stage durations for the roofline come from a second pass of
    # the same steps with the timing on (serial kernel order, `roofline.serial_order_value`).
    chk.setTiming(False)
    step_device(0, warm_ev); torch.cuda.synchronize()
    launches0 = chk.stats()["kernel_launches"]
    # one extra window at the end (N > 1): the exchange of the last step
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps + 1)]
    k0_ms, k1_ms, k2_ms, stage_ms = [], [], [], []
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)               # evict L2 (untimed)
        ev[i][0].record()
        step_device(i, ev[i][0])
        ev[i][1].record()
    ev[args.steps][0].record()
    if world > 1:
        exchange((args.steps - 1) & 1, ev[args.steps][0])
        torch.cuda.current_stream().wait_event(ev_done)
    ev[args.steps][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - wall0
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)
    launches = chk.stats()["kernel_launches"] - launches0      # kernels of this library launched inside the timed region
    if args.dump_outputs and rank == 0:    # the last timed step's outputs, before the passes below overwrite them
        cnt = int(loc_cnt.item())
        outs = {"valid": d_valid.cpu().numpy().astype(np.float32),
                "valid_bits": my_bits[(args.steps - 1) & 1].cpu().numpy().view(np.uint32).astype(np.float64),
                "valid_index": loc_idx[:cnt].cpu().numpy().astype(np.float64),
                "valid_count": np.array([cnt], np.float64)}
        if world > 1:
            outs["all_valid_bits"] = all_bits.cpu().numpy().view(np.uint32).astype(np.float64)
        dump_outputs(args.dump_outputs, outs)
    # second pass, per-stage timing ON (the stages of a round then run one after the other on the call's stream): stage
    # durations from the library's CUDA events, and the throughput of that serial order
    chk.setTiming(True)
    fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    timed_ms = 0.0
    chk.isValidBatchBits(d_poses, d_valid, my_bits[0]); torch.cuda.synchronize()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)
        fa.record()
        chk.isValidBatchBits(d_poses, d_valid, my_bits[0])
        chk.compactValidU32(d_valid, base=rank * n, out_idx=loc_idx, out_cnt=loc_cnt)
        fb.record()
        ka, kb, kc = chk.lastKernelTimesMs()   # waits for this step's kernels (events on the same stream)
        k0_ms.append(ka); k1_ms.append(kb); k2_ms.append(kc); stage_ms.append(chk.lastStageTimesMs())
        torch.cuda.synchronize()
        timed_ms += fa.elapsed_time(fb)
    fork_ms = timed_ms
    # the same step un-pipelined (check -> pack -> local list -> all-gather on one stream)
    sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step_serial(); torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    serial_ms = 0.0
    for i in range(args.steps):
        flush.fill_(i & 0xFF)
        sa.record(); step_serial(); sb.record(); torch.cuda.synchronize()
        serial_ms += sa.elapsed_time(sb)
    exchange_ok = None
    if world > 1:   # verify the WHOLE exchange: every gathered bit against every rank's verdict byte, and the local list
        all_valid = torch.empty(world * n, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(all_valid, d_valid)
        w64 = all_bits.to(torch.int64) & 0xFFFFFFFF
        unpacked = ((w64[:, None] >> torch.arange(32, device="cuda")[None, :]) & 1).reshape(-1).to(torch.uint8)
        want_idx = (torch.nonzero(d_valid).reshape(-1) + rank * n).to(torch.int32)
        cnt = int(loc_cnt.item())
        ok = torch.equal(unpacked, (all_valid != 0).to(torch.uint8)) and cnt == want_idx.numel() and torch.equal(loc_idx[:cnt], want_idx)
        okt = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        exchange_ok = bool(int(okt.item()))
    deferred = chk.stats()["last_deferred"]
    queued = chk.stats()["last_queued_boxes"]
    stats_last = chk.stats()

    # ---- timed region: end to end through the host-buffer C-ABI call ---------------------------
    e2e_steps = args.steps
    chk.setTiming(False)     # per-stage event timing makes the host-fed call run its slices back to back (no copy/compute overlap)
    step_e2e(); step_e2e_f64()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    step_e2e_f64(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e_f64()
    torch.cuda.synchronize()
    e2e64_s = time.perf_counter() - t0
    e2e_mask = hb_valid.array.copy()
    clocks = sampler.stop() if rank == 0 else None
    # Two caller threads, each with its own handle and pinned buffers (what a multi-threaded planner does): the copy of one
    # call overlaps the kernels of the other. Reported beside the single-caller number, never instead of it.
    two_callers = None
    if world == 1:
        try:
            import threading
            chk2 = apb.StateValidityChecker(synth.PARAMS_YAML, device=local)
            chk2.setMap(m); chk2.updateHeightField()
            hb2_p, hb2_v = capi.HostBuffer((n, 7), np.float32), capi.HostBuffer((n,), np.uint8)
            hb2_p.array[:] = hb_poses32.array
            jobs = [(chk, hb_poses32.array.ctypes.data, hb_valid.array.ctypes.data), (chk2, hb2_p.array.ctypes.data, hb2_v.array.ctypes.data)]
            for c_, p_, v_ in jobs:
                c_.isValidHostPtr(p_, n, v_, f32=True)

            def caller(c_, p_, v_):
                for _ in range(e2e_steps):
                    c_.isValidHostPtr(p_, n, v_, f32=True)
            th = [threading.Thread(target=caller, args=j) for j in jobs]
            torch.cuda.synchronize(); t0 = time.perf_counter()
            for t_ in th: t_.start()
            for t_ in th: t_.join()
            torch.cuda.synchronize(); dt2 = time.perf_counter() - t0
            two_callers = {"value": 2 * n * e2e_steps / dt2, "unit": "poses/s", "callers": 2,
                           "masks_equal": bool(np.array_equal(hb2_v.array, e2e_mask) and np.array_equal(hb_valid.array, e2e_mask)),
                           "note": "two threads, one handle + pinned buffer pair each, float32 states; same bytes per call as e2e"}
            del chk2
        except Exception as ex:
            two_callers = {"error": repr(ex)}
    chk.setTiming(True)

    # ---- secondary workloads of the same hot path (BASELINE configs[2] and [3]); N = 1 only, short -------------
    secondary = None
    if world == 1 and args.workload == "c2":
        secondary = {}
        s1, s2 = synth.make_edges(m, 100_000, seed=4)
        d1, d2 = torch.from_numpy(s1).cuda(), torch.from_numpy(s2).cuda()
        mv = apb.MotionValidator(chk, 20)
        ev_out = torch.empty(100_000, dtype=torch.uint8, device="cuda")
        for _ in range(3):
            mv.checkMotionBatch(d1, d2, out=ev_out)
        torch.cuda.synchronize()
        a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            mv.checkMotionBatch(d1, d2, out=ev_out)
        bb.record(); torch.cuda.synchronize()
        ms = a.elapsed_time(bb) / 20
        o_e, kind_e = cpu_oracle(synth.PARAMS_YAML)      # mask of the FULL batch against the compiled reference
        o_e.set_map(m)
        cores_e = min(os.cpu_count() or 1, 32)
        t0 = time.perf_counter(); ev_ref = o_e.check_motions_mt(s1, s2, 20, cores_e); t_e = time.perf_counter() - t0
        secondary["edge_validity"] = {"workload": "configs[2]: 100k edges x 20 interpolation steps (+ end state), same map",
                                      "edges_per_s": 100_000 / (ms * 1e-3), "state_checks_per_s_upper": 2_100_000 / (ms * 1e-3),
                                      "ms_per_batch": ms, "valid_fraction": float(ev_out.float().mean()),
                                      "mask_equals_reference": bool(np.array_equal(ev_out.cpu().numpy(), ev_ref)),
                                      "cpu": {"kind": kind_e, "cores": cores_e, "edges_per_s": 100_000 / t_e,
                                              "sample": "all 100k edges (early exit at the first invalid state)"}}
        del o_e
        try:   # SURVEY 8(d): C2 at a second roughness level -- the regime where most torso boxes reach the plane pass
            from oracle import orc
            m_r = synth.make_fbm_map(MAP_N, MAP_N, MAP_RES, seed=MAP_SEED, **ROUGH_MAP)
            p_r = synth.make_terrain_poses(m_r, n, seed=POSE_SEED, **ROUGH_POSES)
            o_r, kind_r = cpu_oracle(synth.PARAMS_YAML)
            orc.build("port")
            chk_r = apb.StateValidityChecker(synth.PARAMS_YAML, device=local)
            secondary["c2_rough"] = pose_workload(torch, chk_r, flush, m_r, p_r, 20, o_r, kind_r,
                                                  orc.Oracle(synth.PARAMS_YAML, "port"))
            secondary["c2_rough"]["generator"] = {"map": ROUGH_MAP, "poses": ROUGH_POSES, "map_seed": MAP_SEED, "pose_seed": POSE_SEED}
            del chk_r, o_r
        except Exception as ex:
            secondary["c2_rough"] = {"error": repr(ex)}
        try:   # addValidMilestone connection batches (prm_motion_cost.cpp:341-372): per-edge interior-state counts
            e1, e2 = synth.make_edges(m, 200_000, seed=9, dmin=0.05, dmax=3.4)
            g1, g2 = torch.from_numpy(e1).cuda(), torch.from_numpy(e2).cuda()
            mvi = apb.MotionValidator(chk)
            pref, ni = mvi.checkEdgeInteriors(g1, g2)
            torch.cuda.synchronize(); a.record()
            for _ in range(10):
                pref, ni = mvi.checkEdgeInteriors(g1, g2, n_interp=ni)
            bb.record(); torch.cuda.synchronize()
            ms_i = a.elapsed_time(bb) / 10
            secondary["edge_interiors"] = {"workload": "200k candidate connections, n_interp = lateralDistance/0.5 interior states each",
                                           "edges_per_s": 200_000 / (ms_i * 1e-3), "interior_states": int(ni.sum()),
                                           "state_checks_per_s_upper": float(ni.sum()) / (ms_i * 1e-3), "ms_per_batch": ms_i,
                                           "fully_valid_fraction": float((pref == ni).float().mean())}
        except Exception as ex:
            secondary["edge_interiors"] = {"error": repr(ex)}
        plo = apb.PathLengthObjective(chk)
        c_out = torch.empty(100_000, dtype=torch.float64, device="cuda")
        plo.motionCostBatch(d1, d2, out=c_out); torch.cuda.synchronize(); a.record()
        for _ in range(50):
            plo.motionCostBatch(d1, d2, out=c_out)
        bb.record(); torch.cuda.synchronize()
        secondary["path_length_cost"] = {"evals_per_s": 100_000 * 50 / (a.elapsed_time(bb) * 1e-3)}
        try:   # per-map work (the reference: HeightMapBoxChecker::setHeightField = one layer copy per checker at 1 Hz)
            from oracle.basic_oracle import BasicParams
            t_set = []
            for _ in range(4):
                t0 = time.perf_counter(); chk.updateHeightField(); torch.cuda.synchronize(); t_set.append(time.perf_counter() - t0)
            trav, obs = synth.make_traversability(m, seed=13)
            chk.processBasic(m.elevation, trav, obs, m.res, BasicParams())
            t_pb = []
            for _ in range(3):
                t0 = time.perf_counter(); mk, _thr = chk.processBasic(m.elevation, trav, obs, m.res, BasicParams()); t_pb.append(time.perf_counter() - t0)
            secondary["map_update"] = {
                "artp_set_map_ms": 1e3 * min(t_set[1:]), "what_set_map": "H2D of both 1000x1000 layers + column reverse + plane tables "
                "(hash of 2 M triangle planes) + range tables (levels 1-5 / 1-3), through the Python wrapper",
                "artp_process_basic_ms": 1e3 * min(t_pb), "what_process_basic": "processors::Basic masking on the device: 3 layers H2D, "
                "7 morphology passes (elements 3..15 cells), elevation_masked + traversability_thresholded D2H",
                "masked_traversable_fraction": float(np.isfinite(mk).mean())}
        except Exception as ex:
            secondary["map_update"] = {"error": repr(ex)}
        try:   # latency of small batches through the host-buffer API (what a one-state isValid call pays)
            lat = {}
            chk.setTiming(False)   # the one-launch latency path (n <= 16) is bypassed while kernel timing is on
            for nb in (1, 16, 64, 65, 4096, 65536):
                hp = h_poses32[:nb]
                for _ in range(20):
                    chk.isValidHostPtr(hp.data_ptr(), nb, h_valid.data_ptr(), f32=True)
                reps = 200 if nb <= 4096 else 50
                t0 = time.perf_counter()
                for _ in range(reps):
                    chk.isValidHostPtr(hp.data_ptr(), nb, h_valid.data_ptr(), f32=True)
                lat[str(nb)] = (time.perf_counter() - t0) / reps * 1e6
            chk.setTiming(True)
            secondary["host_api_latency_us_by_batch"] = lat
        except Exception as ex:
            secondary["host_api_latency_us_by_batch"] = {"error": repr(ex)}
        try:   # SURVEY 8(f) rows 1-2: device sampler + fused sample -> isValid -> compact (no host pose stream)
            L = synth.make_sampler_layers(m, seed=7)
            smp = apb.SE3FromSE2Sampler(chk, L, synth.sampler_params_for(m), seed=1)
            nd = 1 << 20
            s_out = torch.empty((nd, 7), dtype=torch.float64, device="cuda")
            s_cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
            for _ in range(3):
                smp.sampleValidDevice(nd, 0, s_out, s_cnt)
            torch.cuda.synchronize(); a.record()
            for it in range(20):
                smp.sampleValidDevice(nd, it * nd, s_out, s_cnt)
            bb.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(bb) / 20
            h_out = torch.empty((nd, 7), dtype=torch.float64).pin_memory()
            smp.sampleValidBatch(nd, first=0, out=h_out)
            t0 = time.perf_counter()
            for it in range(10):
                hs, nv = smp.sampleValidBatch(nd, first=it * nd, out=h_out)
            host_s = (time.perf_counter() - t0) / 10
            secondary["fused_sample_check_compact"] = {
                "workload": "2^20 candidates drawn from the map's sampling CDF on the device (Philox stream), checked, valid ones compacted in draw order",
                "candidates_per_s_device": nd / (ms * 1e-3), "ms_per_batch": ms, "valid_fraction": nv / nd,
                "candidates_per_s_host_api": nd / host_s, "d2h_bytes_per_batch": int(nv) * 56, "h2d_bytes_per_batch": 0}
        except Exception as ex:
            secondary["fused_sample_check_compact"] = {"error": repr(ex)}
        try:
            from art_planner_b200 import costnet
            m4 = synth.make_fbm_map(256, 256, MAP_RES, seed=MAP_SEED, amp=0.6)
            chk4 = apb.StateValidityChecker(synth.PARAMS_YAML, device=local)
            chk4.setMap(m4); chk4.updateHeightField()
            mco = apb.MotionCostObjective(chk4)
            mco.setWeights(costnet.make_state_dict(seed=5))
            tms = []
            for _ in range(8):
                mco.updateFeatures(); tms.append(mco.lastTrunkTimesMs())
            tms = np.array(tms[3:]).mean(0)
            qd = torch.from_numpy(costnet.make_queries(m4, 4096, seed=6)).cuda()
            qo = torch.empty((4096, 3), dtype=torch.float32, device="cuda")
            for _ in range(3):
                mco.costQuery(qd, out=qo)
            torch.cuda.synchronize(); a.record()
            for _ in range(100):
                mco.costQuery(qd, out=qo)
            bb.record(); torch.cuda.synchronize()
            hms = a.elapsed_time(bb) / 100
            secondary["motion_cost_cnn"] = {
                "workload": "configs[3]: 256x256 elevation patch -> cost CNN trunk, 4096-query batch, seeded random weights",
                "trunk_ms": float(tms[2]), "conv3x3_stack_ms": float(tms[0]), "conv15x15_tcgen05_ms": float(tms[1]),
                "trunk_tflops": 13.41e9 / (float(tms[2]) * 1e-3) / 1e12, "conv15_tflops": 11.21e9 / (float(tms[1]) * 1e-3) / 1e12,
                "head_ms_4096_queries": hms, "edge_cost_evals_per_s": 4096 / (hms * 1e-3)}
        except Exception as ex:   # never let a secondary workload take the headline line down
            secondary["motion_cost_cnn"] = {"error": repr(ex)}

    c5 = None
    try:
        c5 = run_c5(torch, dist, apb, synth, world, rank, local, flush)
    except Exception as ex:      # never let the sharded workload take the headline line down
        c5 = {"error": repr(ex)}
    t = torch.tensor([dev_ms, e2e_s * 1e3, serial_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, serial_ms = float(t[0]), float(t[1]), float(t[2])
    valid_ref = None

    if rank == 0:
        value = world * n * args.steps / (dev_ms * 1e-3)
        e2e_value = world * n * e2e_steps / (e2e_ms * 1e-3)
        # ---- CPU baseline + algorithmic bytes from the oracle on a bounded sample ---------------
        o, kind = cpu_oracle(synth.PARAMS_YAML)
        o.set_map(m)
        # one ODE world + two layer copies per thread: the probe bounds host memory on big maps
        n1 = 20_000
        t0 = time.perf_counter(); v1 = o.check_poses(poses[:n1]); t_single = time.perf_counter() - t0
        got = d_valid.cpu().numpy()
        e2e_mask_ok = bool(np.array_equal(e2e_mask, got))   # the host-fed (sliced) path returns the device path's mask
        if world == 1:   # the timed all-threads CPU baseline belongs to the N = 1 line only
            cores = best_thread_count(o, poses, os.cpu_count() or 1, m.rows * m.cols > 4_000_000)
            n_mt = 400_000
            o.check_poses_mt(poses[:cores * 64], cores)   # builds the per-thread ODE worlds (one-time per map, untimed)
            t0 = time.perf_counter(); v_mt = o.check_poses_mt(poses[:n_mt], cores); t_mt = time.perf_counter() - t0
            parity_ok = bool(np.array_equal(got[:n_mt], v_mt) and np.array_equal(got[:n1], v1))
            cpu_baseline = {"value": n_mt / t_mt, "unit": "poses/s", "cores": cores, "kind": kind,
                            "sample": f"first {n_mt} poses of the workload, {cores} threads (best of a probe over 8..{os.cpu_count()}); single-thread on first {n1}",
                            "single_thread_value": n1 / t_single, "mask_equals_gpu": parity_ok}
        else:
            cpu_baseline = {"value": None, "unit": "poses/s", "cores": 1, "kind": kind,
                            "sample": f"N > 1: not timed (see the N = 1 line); rank 0's mask checked against the oracle on its first {n1} poses",
                            "single_thread_value": n1 / t_single, "mask_equals_gpu": bool(np.array_equal(got[:n1], v1))}
        from oracle import orc
        orc.build("port")
        port = orc.Oracle(synth.PARAMS_YAML, "port")
        port.set_map(m)
        _, zv = port.check_poses(poses[:50_000], want_zone=True)
        bytes_per_pose = 56.0 + 1.0 + 4.0 * float(zv.mean())
        peak, peak_src = load_peaks()
        # Roofline bookkeeping (DESIGN.md 4.2): the algorithmic bytes belong to the whole pass (classify + the two box
        # queues + grouping), so they are divided by the SUM of the stage durations; the dominant kernel is the reach-box
        # queue launch of box_tiles_warp_kernel.
        sm = np.mean(np.array(stage_ms), 0)
        k0, k_torso, k_reach, k2 = float(sm[0]), float(sm[1]), float(sm[2] + sm[3]), float(sm[4])
        pass_ms = k0 + k_torso + k_reach + k2
        achieved = bytes_per_pose * n / (pass_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("reach_queues_dram_bytes_per_pass")   # group kernel + one-warp-per-box launch
        port_mix = exit_mix(port, poses[:20_000])
        out = {
            "metric": "pose-validity checks/s", "value": value, "unit": "poses/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if args.workload == "c2" else
                       "configs[4]: fBm 4000x4000@0.04m map, 1M samples per GPU inside the GPU's spatial slab, yaml robot geometry",
                       "poses_per_gpu": n, "map": f"{m.rows}x{m.cols}@{MAP_RES}", "map_generator": m.desc,
                       "roughness": "gentle level of SURVEY 8(d) by its exit mix (torso: %.0f %% above the zone, %.1f %% through the full triangle / plane pass); the rough level is secondary.c2_rough" % (100 * port_mix["torso"]["above"], 100 * port_mix["torso"]["fall_through"]),
                       "exit_mix": port_mix,
                       "map_seed": MAP_SEED, "pose_seed": POSE_SEED, "l2": "flushed between timed steps (256 MiB write)",
                       "step": "isValid of the batch (verdict bytes) + bit-packed verdicts + the ordered 32-bit index list of the valid samples",
                       "parallelism": f"pose shards x{world}, replicated 1000x1000 map" + (", one NCCL all-gather of bit-packed masks per step, pipelined: the exchange of step i runs on a side stream inside the timed window of step i+1 (+ one closing window); see exchange.unpipelined_value and c5 (spatial shards)" if world > 1 else "")},
            "e2e": {"value": e2e_value, "unit": "poses/s", "h2d_bytes_per_step": n * 28, "d2h_bytes_per_step": n, "mask_equals_device_path": e2e_mask_ok,
                    "ms_per_step": e2e_ms / e2e_steps, "api": "artp_check_poses_f32 (states cast to float by the adapter while it gathers them, exact), buffers from artp_host_alloc",
                    "f64_api_value": world * n * e2e_steps / e2e64_s, "f64_api_h2d_bytes_per_step": n * 56, "two_callers": two_callers,
                    "note": "PCIe Gen5 x16 moves 53-55 GB/s here (profiles/pcie_probe.cu): 28 MB = 0.52 ms, 56 MB = 1.04 ms, so the double entry point is copy-bound at <= 0.96e9 poses/s"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "reach_groups_kernel + box_tiles_warp_kernel (the two reach-box queues)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_pose": bytes_per_pose, "kernel_ms": k_reach,
                         "classify_kernel_ms": k0, "torso_queue_kernel_ms": k_torso, "group_kernel_ms": k2, "pass_ms": pass_ms,
                         "serial_order_value": world * n * args.steps / (fork_ms * 1e-3),
                         "stage_times_from": "a second pass of the same steps with artp_set_timing on: the stages then run one after the other on one stream (their CUDA events need that); the timed region runs the shipped default, the three box kernels of a round side by side",
                         "queued_boxes": int(queued), "deferred_boxes": int(deferred),
                         "stage_ms": dict(zip(("classify", "torso_queue", "reach_queue_warp", "reach_queue_groups", "group"), [float(x) for x in sm])),
                         "queued_warp_stage": stats_last["last_queued_warp_stage"],
                         "queued_reach_stage": stats_last["last_queued_reach_stage"],
                         "queued_reach_groups": stats_last["last_reach_plane_stage"],
                         "actual_dram_GBps_dominant_kernel": (traffic / (k_reach * 1e-3) / 1e9) if traffic else None,
                         "note": "achieved = ALGORITHMIC bytes (the zone vertices the reference scans, SURVEY 8d) / sum of the stage "
                                 "durations; the range tables, plane tables and vertex probes answer most of those scans without reading "
                                 "them, so frac exceeds 1 while real DRAM traffic (traffic, ncu) stays near 1 % of peak: the pipeline is "
                                 "instruction-issue bound (group kernel: 68 % of issue slots busy, 20 of 32 lanes; profiles/r02_v6_*)"},
            "cpu_baseline": cpu_baseline,
            "clocks": clocks, "wall_s_timed_region": wall, "secondary": secondary, "exchange_ok": exchange_ok,
            "exchange": {"unpipelined_value": world * n * args.steps / (serial_ms * 1e-3), "unpipelined_ms_per_step": serial_ms / args.steps,
                         "wire_bytes_per_rank_per_step": n // 8 if world > 1 else 0,
                         "what": "check + pack + this shard's ordered 32-bit index list" + (" + one NCCL all-gather of the bit masks" if world > 1 else "")},
            "c5": c5,
        }
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
