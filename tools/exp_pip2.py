"""Round-2 PIP experiments on one B200: build time, query time, raster census for the config-2 workload.
One JSON line per run.

  python tools/exp_pip2.py [--points N] [--polys M --grid G] [--reps R] [--tag TAG]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from geopolars_b200 import GeoArrowArray, synth
from geopolars_b200 import engine as E

ap = argparse.ArgumentParser()
ap.add_argument("--points", type=int, default=100_000_000)
ap.add_argument("--polys", type=int, default=10_000)
ap.add_argument("--grid", type=int, default=100)
ap.add_argument("--cell", type=float, default=10.0)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--tag", default="")
ap.add_argument("--outside", action="store_true", help="shift the points outside the grid: the streaming floor")
ap.add_argument("--count", action="store_true")
args = ap.parse_args()

dev = torch.device("cuda", 0)
st = torch.cuda.Stream()
n = args.points
with torch.cuda.stream(st):
    ctx = E.Context(0, st.cuda_stream)
    pts = torch.empty((n, 2), dtype=torch.float64, device=dev)
    E.check(ctx.lib.gpl_gen_uniform_points(ctx._h, 2, 0, n, args.grid * args.cell, pts.data_ptr()))
    if args.outside:
        pts += 5.0 * args.grid * args.cell
    ids = torch.empty(n, dtype=torch.int32, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev) if args.count else None
    xy, ro, go = synth.star_polygons(args.polys, args.grid, args.cell)
    polys = ctx.upload(GeoArrowArray.polygons(xy, ro, go))
    st.synchronize()
    # build: wall clock around the call + a stream sync (it has one host round trip inside)
    builds = []
    idx = None
    for _ in range(args.reps + 2):
        if idx is not None:
            idx.free()
        st.synchronize()
        t0 = time.perf_counter()
        idx = E.PipIndex(polys)
        st.synchronize()
        builds.append(1e3 * (time.perf_counter() - t0))
    builds = builds[2:]
    stats = idx.stats()
    phases = idx.phases()
    q = []
    for _ in range(args.reps + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        idx.query_device(pts.data_ptr(), n, ids.data_ptr(), cnt.data_ptr() if cnt is not None else 0)
        e1.record(st)
        st.synchronize()
        q.append(e0.elapsed_time(e1))
    q = q[2:]
    stats = idx.stats()
    hits = int((ids >= 0).sum().item())
    # order-sensitive checksum of the id column, to compare variants across processes
    w = torch.arange(1, 1025, device=dev, dtype=torch.int64).repeat((n + 1023) // 1024)[:n]
    checksum = int(((ids.to(torch.int64) + 2) * w).sum().item())
    fg = stats["fine_cells_per_axis"]
    line = {
        "tag": args.tag, "points": n, "polys": args.polys,
        "build_ms_min": min(builds), "build_ms_mean": sum(builds) / len(builds),
        "query_ms_min": min(q), "query_ms_mean": sum(q) / len(q),
        "read_GBps": 16.0 * n / (min(q) * 1e-3) / 1e9,
        "hit_rate": hits / n, "checksum": checksum, "index_MB": stats["bytes"] / 1e6,
        "raster_log2": stats["raster_log2"], "fine_cells_per_axis": fg,
        "walk_cell_frac": stats["raster_walk_cells"] / max(1, fg * fg), "inside_cell_frac": stats["raster_inside_cells"] / max(1, fg * fg),
        "fill_phases_us": [round(v, 1) for v in phases],
        "deferred_per_query": stats["deferred"] / (args.reps + 2), "parts_not_fast": stats["parts_not_fast"],
    }
    print(json.dumps(line), flush=True)
