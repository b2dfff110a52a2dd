"""Map change detection + roadmap invalidation on the device vs the single-thread CPU restatement.

    python profiles/roadmap_update.py --out DIR [--reps 50] [--skip-4000]

Workloads (DESIGN 4.6):
  1000   a 1000^2 @ 0.04 m map pair shifted by a non-integer number of cells (synth.make_map_pair), 10 000 vertices and
         50 000 edges between vertices less than 1.5 m apart (synth.make_roadmap: numpy grid binning)
  4000   a 4000^2 @ 0.04 m pair, 100 000 vertices, 10^6 edges
Per workload: artp_compute_change from host layers (blocking call: 4 layers H2D + the float layer D2H) and from device
layers (CUDA events over --reps back-to-back calls, bit layer only and with the float layer); artp_roadmap_updates
through the host API (blocking) and the device API (events); the CPU oracle (orc_compute_change, orc_roadmap_updates)
single-threaded, without and with the reference's per-edge copy of the `updated` layer (map.cpp:46; on a stated prefix
of the edges when the full run would take too long); and whether every GPU output equals the CPU one. Device name and
power limit are read in the same run. Writes DIR/roadmap_update.json and prints it. Needs a CUDA device: no fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

THR = 0.1   # params.yaml: lazy_prm_star_min_update.height_change_for_update


def device_info():
    import torch
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001 - reported, not fatal
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def host_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def device_ms(fn, reps):
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def torch_layers(m):
    import torch
    import types
    f = lambda x: torch.from_numpy(np.ascontiguousarray(np.asarray(x, np.float32).T)).cuda().t()
    return types.SimpleNamespace(elevation=f(m.elevation), traversability_thresholded=f(m.traversability_thresholded),
                                 res=m.res, cx=m.cx, cy=m.cy)


def run(name, rows, nv, ne, octaves, faithful_prefix, reps):
    import torch
    import art_planner_b200 as ap
    from art_planner_b200 import synth
    from oracle import roadmap_orc as orc
    t0 = time.perf_counter()
    new, old = synth.make_map_pair(seed=11, index=0, rows=rows, cols=rows, res=0.04, thr=THR, octaves=octaves)
    states, edges = synth.make_roadmap(old, nv, ne, seed=12, max_dist=1.5)
    gen_s = time.perf_counter() - t0
    chk = ap.StateValidityChecker(synth.PARAMS_YAML, device=0)
    r = {"map": f"{rows}x{rows}@0.04", "shift_cells": [new.cx / 0.04, new.cy / 0.04], "n_vertices": int(len(states)),
         "n_edges": int(len(edges)), "generate_s": round(gen_s, 2)}
    # ---- change --------------------------------------------------------------------------------------------------
    upd_gpu = chk.computeChange(new, old, THR)
    r["change_host_ms_median_min"] = host_ms(lambda: chk.computeChange(new, old, THR), max(5, reps // 5))
    r["change_host_bits_only_ms_median_min"] = host_ms(lambda: chk.computeChange(new, old, THR, want_layer=False),
                                                        max(5, reps // 5))
    dn, do = torch_layers(new), torch_layers(old)
    out = torch.empty((rows, rows), dtype=torch.float32, device="cuda").t()
    r["change_device_bits_ms"] = device_ms(lambda: chk.computeChange(dn, do, THR, want_layer=False), reps)
    r["change_device_bits_and_float_ms"] = device_ms(lambda: chk.computeChange(dn, do, THR, out=out), reps)
    torch.cuda.synchronize()
    cells = rows * rows
    r["change_device_bytes"] = cells * (4 * 4 + 1 / 8)          # four float layers read, one bit written
    r["change_device_GBps"] = r["change_device_bytes"] / (r["change_device_bits_ms"] * 1e-3) / 1e9
    t = time.perf_counter()
    upd_cpu, ok = orc.compute_change(new, old, THR)
    r["change_cpu_ms"] = (time.perf_counter() - t) * 1e3
    r["change_overlap_ok"] = bool(ok)
    r["updated_fraction"] = float(upd_cpu.mean())
    change_equal = (np.array_equal(upd_gpu.view(np.uint32), upd_cpu.view(np.uint32)) and
                    np.array_equal(out.cpu().numpy().view(np.uint32), upd_cpu.view(np.uint32)))
    # ---- roadmap -------------------------------------------------------------------------------------------------
    chk.computeChange(dn, do, THR, want_layer=False)
    vf, ef = chk.roadmapUpdates(states, edges)
    r["roadmap_host_ms_median_min"] = host_ms(lambda: chk.roadmapUpdates(states, edges), max(5, reps // 5))
    ds = torch.from_numpy(states).cuda()
    de = torch.from_numpy(edges.astype(np.int32)).cuda()
    ov = torch.empty(len(states), dtype=torch.uint8, device="cuda")
    oe = torch.empty(len(edges), dtype=torch.uint8, device="cuda")
    r["roadmap_device_ms"] = device_ms(lambda: chk.roadmapUpdates(ds, de, ov, oe), reps)
    torch.cuda.synchronize()
    chk.pollError()
    r["roadmap_launches_per_call"] = chk.stats()["last_launches"]
    t = time.perf_counter()
    cvf, cef = orc.roadmap_updates(new, upd_cpu, states, edges)
    r["roadmap_cpu_ms"] = (time.perf_counter() - t) * 1e3
    k = min(faithful_prefix, len(edges))
    t = time.perf_counter()
    fvf, fef = orc.roadmap_updates(new, upd_cpu, states, edges[:k], copy_layer_per_edge=True)
    fs = time.perf_counter() - t
    r["roadmap_cpu_layer_copy"] = {"edges_timed": int(k), "ms": fs * 1e3,
                                   "ms_per_edge": fs * 1e3 / max(k, 1),
                                   "ms_extrapolated_to_all_edges": fs * 1e3 / max(k, 1) * len(edges)}
    r["vertex_flag_counts"] = np.bincount(cvf, minlength=3).tolist()
    r["edge_flag_counts"] = np.bincount(cef, minlength=3).tolist()
    roadmap_equal = (np.array_equal(vf, cvf) and np.array_equal(ef, cef) and np.array_equal(ov.cpu().numpy(), cvf) and
                     np.array_equal(oe.cpu().numpy(), cef) and np.array_equal(fvf, cvf) and np.array_equal(fef, cef[:k]))
    r["outputs_equal"] = bool(change_equal and roadmap_equal)
    return r


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", required=True)
    ap_.add_argument("--reps", type=int, default=50)
    ap_.add_argument("--skip-4000", action="store_true")
    a = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("roadmap_update.py needs a CUDA device")
    from art_planner_b200 import build
    from oracle import roadmap_orc
    build.build()
    roadmap_orc.build()
    res = {"device": device_info(), "threshold": THR,
           "note": "device times: CUDA events over back-to-back calls after warm-up; host times: perf_counter around "
                   "blocking calls; CPU: one thread of the GPU host. The 4000^2 change inputs (256 MB) exceed L2; the "
                   "roadmap's bit layer (2 MB) stays in L2 across calls.",
           "workloads": {}}
    res["workloads"]["1000"] = run("1000", 1000, 10_000, 50_000, 4, 5000, a.reps)
    if not a.skip_4000:
        res["workloads"]["4000"] = run("4000", 4000, 100_000, 1_000_000, 3, 200, a.reps)
    res["outputs_equal"] = all(w["outputs_equal"] for w in res["workloads"].values())
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "roadmap_update.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
