#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the GeoSeries hot path.

Default workload `c2` (BASELINE.json configs[1], the configuration `metric` is quoted on): N_POINTS uniform random
points `.contains()`-joined against 10 000 64-vertex star polygons (SURVEY.md §8d config 2), one such batch per GPU
(weak scaling: every rank owns its own 100 M-point row range, the polygon side is broadcast from rank 0 over NCCL —
the only exchange step this path has).

One "step" = one pass of the hot path over one batch: [N>1: NCCL broadcast of the polygon coordinates] + polygon
index build + the point-in-polygon kernel over all of the rank's points + the per-polygon hit counts [+ N>1: all-reduce
of the counts].  `value` = points processed by all ranks / max-over-ranks device time,
inputs resident in HBM.  `e2e` = the same join through the C ABI from pinned HOST buffers (H2D of the points and D2H
of the ids inside the timed region, chunked and overlapped).

Other BASELINE configurations are separate arms (`--workload`), same JSON contract, same verification rules:
  c3  50 M LineString pairs (K = 16): euclidean distance + intersects, rows sharded over the ranks (strong scaling)
  c4  125 M points per GPU x 1 000 polygons: join + counts all-reduce + the id column GATHERED to rank 0 (weak; 1 B points at N=8)
  c5  10 M 257-coordinate polygons: convex_hull + affine_transform, rows sharded (strong scaling), hull rings gathered to rank 0

After the timed region every rank checks its results against the CPU oracle on a bounded slice (`verify` in the JSON
line) — a number whose results differ from the reference's is not printed at all.

Timing: W (>= 3) warm-up steps, extended with further untimed steps until the device has been under this load for
MIN_LOAD_S (`config.warmup_steps_run`; nvidia-smi needs that long to deliver `clocks` samples under load — the default timed
region lasts ~6 ms), then EXACTLY K steps between two CUDA events on the context's stream, barrier + synchronize on both
sides, max over ranks.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
  python bench.py --impl reference      # the CPU restatement of the reference path on the host cores
  python bench.py --dump-outputs bench_outputs   # + what the last timed step computed, as .npy files

`--dump-outputs DIR` writes, after the timed steps, the arrays the last timed step handed its caller on rank 0, as float64
DIR/<name>.npy: whole when small, else at a fixed sample of rows (seed 0, `rows.npy`), at most DUMP_BYTES in all.  The
inputs are generated from fixed seeds, so two builds of the project can be compared output for output.

The CPU oracle (oracle/) is used here only for `cpu_baseline`, `--impl reference` and the post-run verification; the
measured GPU path never touches it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it

METRIC = "geometries/s"
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this many bytes
MIN_LOAD_S = 0.6  # seconds of warm-up load before the timed region (so that the nvidia-smi clock sampler has samples under load)
COORD_BYTES = 16  # one f64 xy pair: the algorithmic bytes per coordinate (SURVEY.md §8d)


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def recorded_traffic(name):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, if any"""
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            with open(p) as f:
                return json.load(f)
        except Exception:
            return None
    return None


def all_cpus():
    return sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))


def sample_rows(n, k, device):
    """row numbers of a --dump-outputs sample: all n rows when n <= k, else k distinct rows drawn with seed 0, ascending"""
    import torch

    if n <= k:
        return torch.arange(n, device=device)
    rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    return torch.from_numpy(rows).to(device)


def write_outputs(directory, arrays):
    """--dump-outputs: one float64 DIR/<name>.npy per array"""
    arrays = {k: np.ascontiguousarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte budget"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.t = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for ln in self.proc.stdout:
                self.lines.append(ln.strip())

        self.t = threading.Thread(target=pump, daemon=True)
        self.t.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)  # one more report after the timed region ended
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower() == "active":
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# NUMA placement (multi-GPU end-to-end): a rank's pinned host buffers should live on its GPU's socket
# ------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank: int):
    """Restrict this process to the CPUs of the NUMA node its GPU hangs off, so that pinned buffers are first-touched
    there.  Returns (node, previous affinity) or (None, previous affinity) when the topology cannot be read."""
    prev = set(all_cpus())
    try:
        path = None
        try:
            import torch

            pr = torch.cuda.get_device_properties(local_rank)
            path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/numa_node"
            if not os.path.exists(path):
                path = None
        except Exception:
            path = None
        if path is None:  # NVML reports the bus id as a string
            import pynvml

            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            path = f"/sys/bus/pci/devices/{bus.lower()[-12:]}/numa_node"
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return None, prev
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                if "-" in part:
                    a, b = part.split("-")
                    cpus.update(range(int(a), int(b) + 1))
                elif part:
                    cpus.add(int(part))
        cpus &= prev
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node, prev
    except Exception:
        pass
    return None, prev


# ------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------
class JoinWorkload:
    """c2 / c4: points-in-polygons broadcast join (spatial_index.rs:37-204)"""

    def __init__(self, name, args, env):
        self.name, self.args, self.env = name, args, env
        if name == "c2":
            self.n_polys, self.grid, self.cell, self.nvert = 10_000, 100, 10.0, 64
            self.n = args.points or 100_000_000
            self.gather = False
            self.baseline = "BASELINE configs[1]; SURVEY.md config 2 generator"
        else:
            self.n_polys, self.grid, self.cell, self.nvert = 1_000, 32, 31.25, 64
            self.n = args.points or 125_000_000
            self.gather = True
            self.baseline = "BASELINE configs[3]; SURVEY.md config 4 generator (1 B points at 8 GPUs)"
        self.unit_name = "points"
        self.scaling = "weak"
        self.kernel = "k_pip_stream<LEAN>"
        self.traffic_file = "r2_pip_traffic.json"

    # --- inputs resident in HBM ---------------------------------------------------------------------------
    def setup(self):
        import torch

        from geopolars_b200 import synth
        from geopolars_b200 import engine as E

        e = self.env
        n, m, nv = self.n, self.n_polys, self.nvert
        self.pts = torch.empty((n, 2), dtype=torch.float64, device=e.dev)
        E.check(e.ctx.lib.gpl_gen_uniform_points(e.ctx._h, 2, e.rank * n, n, self.grid * self.cell, self.pts.data_ptr()))
        self.n_pc = m * (nv + 1)
        self.poly_xy = torch.empty((self.n_pc, 2), dtype=torch.float64, device=e.dev)
        self.ring_off = torch.arange(m + 1, dtype=torch.int64, device=e.dev) * (nv + 1)
        self.geom_off = torch.arange(m + 1, dtype=torch.int64, device=e.dev)
        if e.rank == 0:
            xy, _, _ = synth.star_polygons(m, self.grid, self.cell, nv)  # host: libm cos/sin, see synth.py
            self.poly_xy.copy_(torch.from_numpy(xy))
        self.ids = torch.empty(n, dtype=torch.int32, device=e.dev)
        # one zeroed counts column per timed step: no fill kernel inside the timed region.  Warm-up steps cycle through the
        # first n_warm columns (the warm-up may be extended for the clock sampler, see _main); their counts are never read.
        self.counts_pool = torch.zeros((e.total_steps, m), dtype=torch.int64, device=e.dev)
        self.n_warm = max(1, e.total_steps - self.args.steps)
        self.timed_no = 0
        self.gathered = None
        if self.gather and e.world > 1 and e.rank == 0:
            self.gathered = [torch.empty(n, dtype=torch.int32, device=e.dev) for _ in range(e.world)]
        self.idx = None
        self.step_no = 0
        self.units_per_rank = n
        self.algo_bytes = n * COORD_BYTES + self.n_pc * COORD_BYTES  # coordinate bytes read by one launch (SURVEY.md §8d)
        self.write_bytes = 4 * n

    def make_index(self):
        from geopolars_b200 import GeometryType
        from geopolars_b200 import engine as E

        e = self.env
        polys = e.ctx.wrap_device(GeometryType.POLYGON, self.n_polys, self.n_pc, self.poly_xy.data_ptr(), geom_off_ptr=self.geom_off.data_ptr(),
                                  ring_off_ptr=self.ring_off.data_ptr(), n_rings=self.n_polys,
                                  keepalive=(self.poly_xy, self.geom_off, self.ring_off))
        return E.PipIndex(polys)

    def step(self, events):
        import torch
        import torch.distributed as dist

        e = self.env
        if e.world > 1:
            dist.broadcast(self.poly_xy, src=0)  # the broadcast-join's one exchange step (NCCL over NVLink)
        if self.idx is not None:
            self.idx.free()
        self.idx = self.make_index()
        if events is None:
            counts = self.counts_pool[self.step_no % self.n_warm]
        else:
            counts = self.counts_pool[self.n_warm + self.timed_no]
            self.timed_no += 1
        self.step_no += 1
        if events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(e.stream)
        self.idx.query_device(self.pts.data_ptr(), self.n, self.ids.data_ptr())
        if events is not None:
            e1.record(e.stream)
            events.append((e0, e1))
        from geopolars_b200 import engine as E

        E.check(e.ctx.lib.gpl_join_histogram(e.ctx._h, self.ids.data_ptr(), self.n, counts.data_ptr(), self.n_polys, E.GPL_DEVICE))
        if e.world > 1:
            dist.all_reduce(counts)
            if self.gather:
                dist.gather(self.ids, self.gathered if e.rank == 0 else None, dst=0)
        self.last_counts = counts

    def describe_step(self):
        e = self.env
        s = ("NCCL broadcast of polygon coords + " if e.world > 1 else "") + "polygon index build (2 cooperative launches) + " \
            "point-in-polygon kernel over all points + per-polygon hit counts (histogram of the id column)"
        if e.world > 1:
            s += " + counts all-reduce" + (" + id column gathered to rank 0" if self.gather else "")
        return s

    def workload_text(self):
        return f"{self.n} random points per GPU .contains() x {self.n_polys} {self.nvert}-vertex polygons ({self.baseline})"

    def outputs(self):
        """the id column (first containing polygon, -1 for none) at sampled rows, and every per-polygon hit count.  With
        the column gathered (c4 on several GPUs) rank 0 holds every rank's rows: rank r's rows follow as r * n + row."""
        import torch

        segments = self.gathered or [self.ids]
        n = self.n
        rows = sample_rows(n * len(segments), 2_000_000, self.env.dev)
        ids = torch.cat([seg[rows[(rows >= r * n) & (rows < (r + 1) * n)] - r * n] for r, seg in enumerate(segments)])
        return {"rows": rows, "ids": ids, "counts": self.last_counts}

    # --- correctness, outside the timed region ----------------------------------------------------------------
    def verify(self):
        import torch
        import torch.distributed as dist

        from geopolars_b200 import synth
        from oracle import oracle as og

        e = self.env
        m = min(self.n, self.args.verify_rows)
        xy, ro, go = synth.star_polygons(self.n_polys, self.grid, self.cell, self.nvert)
        polys = og.OGArray(og.POLYGON, xy, geom_off=go, ring_off=ro)
        assert np.array_equal(self.poly_xy.cpu().numpy(), xy), "broadcast polygons differ from the generator"
        host_pts = self.pts[:m].cpu().numpy()
        assert np.array_equal(host_pts, og.gen_uniform_points(2, e.rank * self.n, m, self.grid * self.cell)), "device RNG differs from the host RNG"
        want, _ = og.contains_join(polys, host_pts, True, len(all_cpus()))
        got = self.ids[:m].cpu().numpy()
        assert np.array_equal(got, want), f"rank {e.rank}: ids differ from the oracle on the first {m} rows"
        out = {"ids_rows_checked_per_rank": m, "ids_equal_oracle": True, "hit_rate_slice": float((want >= 0).mean())}
        # per-polygon counts: the all-reduced column against an independent bincount of every rank's ids
        ref = torch.bincount(self.ids[self.ids >= 0].to(torch.int64), minlength=self.n_polys)
        if e.world > 1:
            dist.all_reduce(ref)
        assert torch.equal(ref, self.last_counts), f"rank {e.rank}: all-reduced hit counts differ from bincount(ids)"
        out["counts_equal_bincount"] = True
        out["hits_all_ranks"] = int(ref.sum().item())
        st = self.idx.stats()
        out["exact_reevaluations_per_step"] = st["deferred"]
        out["raster"] = {"fine_cells_per_axis": st["fine_cells_per_axis"], "walk_cell_fraction": st["raster_walk_cells"] / max(1, st["fine_cells_per_axis"] ** 2)}
        assert 0 < st["deferred"] < 0.01 * self.n, f"deferred counter {st['deferred']} outside (0, 1 %)"
        if self.gather and e.world > 1:
            # rank 0: every rank's segment of the gathered column against the oracle on that rank's first rows
            if e.rank == 0:
                k = min(self.n, max(1, self.args.verify_rows // e.world))
                for r in range(e.world):
                    pr = og.gen_uniform_points(2, r * self.n, k, self.grid * self.cell)
                    wr, _ = og.contains_join(polys, pr, True, len(all_cpus()))
                    assert np.array_equal(self.gathered[r][:k].cpu().numpy(), wr), f"gathered ids of rank {r} differ from the oracle"
                assert torch.equal(self.gathered[0], self.ids)
                out["gathered_rows_checked_per_rank"] = k
            out["gathered_equal_oracle"] = True
        return out

    # --- end to end: host buffers through the C ABI ---------------------------------------------------------------
    def e2e_setup(self):
        import torch

        self.host_pts = torch.empty((self.n, 2), dtype=torch.float64, pin_memory=True)
        self.host_ids = torch.empty(self.n, dtype=torch.int32, pin_memory=True)
        self.host_pts.copy_(self.pts)
        torch.cuda.synchronize()
        self.poly_host = self.poly_xy.cpu().numpy()
        self.ro_h, self.go_h = self.ring_off.cpu().numpy(), self.geom_off.cpu().numpy()
        self.h2d = self.n * COORD_BYTES + self.n_pc * COORD_BYTES + 8 * 2 * (self.n_polys + 1)
        self.d2h = self.n * 4
        self.e2e_path = "gpl_array_from_buffers(host) + gpl_pip_index_build + gpl_contains_join_host (pinned host points -> pinned host ids)"

    def e2e_step(self):
        from geopolars_b200 import GeoArrowArray
        from geopolars_b200 import engine as E

        arr = GeoArrowArray.polygons(self.poly_host, self.ro_h, self.go_h)
        d_polys = self.env.ctx.upload(arr)  # H2D of the polygon side from host memory
        idx = E.PipIndex(d_polys)
        idx.query_host_pipelined(self.host_pts.data_ptr(), self.n, self.host_ids.data_ptr())
        return idx

    def e2e_check(self):
        import torch

        assert torch.equal(self.host_ids, self.ids.cpu()), "e2e ids differ from the resident run"

    # --- CPU arm -------------------------------------------------------------------------------------------
    def cpu_sample(self, n_sample, threads):
        from geopolars_b200 import synth
        from oracle import oracle as og

        xy, ro, go = synth.star_polygons(self.n_polys, self.grid, self.cell, self.nvert)
        polys = og.OGArray(og.POLYGON, xy, geom_off=go, ring_off=ro)
        pts = og.gen_uniform_points(2, 0, n_sample, self.grid * self.cell)
        og.contains_join(polys, pts[: min(n_sample, 100_000)], True, threads)  # warm-up (page-in, thread pool)
        t0 = time.perf_counter()
        og.contains_join(polys, pts, True, threads)
        dt = time.perf_counter() - t0
        return n_sample / dt, dt, (f"{n_sample} of {self.n} points x {self.n_polys} polygons, bbox-grid candidates + exact test over all "
                                   f"{self.nvert + 1} ring coordinates per candidate (the reference architecture: rstar candidates + geo contains), OpenMP static row chunks")

    def default_cpu_sample(self):
        return 32_000_000


class PairsWorkload:
    """c3: row-wise euclidean distance + intersects over LineString pairs (geoseries.rs:141-146, spatial_index.rs:102-104)"""

    K = 16

    def __init__(self, name, args, env):
        self.name, self.args, self.env = name, args, env
        self.total = args.points or 50_000_000
        self.unit_name = "pairs"
        self.scaling = "strong"
        self.kernel = "k_ls_ls_fast<1> distance + k_ls_ls_fast<0> intersects (+ k_ls_ls_exact)"
        self.traffic_file = "r2_pairs_traffic.json"

    def setup(self):
        import torch

        from geopolars_b200 import GeometryType
        from geopolars_b200 import dist as gd
        from geopolars_b200 import engine as E

        e = self.env
        lo, hi = gd.shard_rows(self.total, e.world, e.rank)
        n, k = hi - lo, self.K
        self.lo, self.n = lo, n
        dev, lib, ctx = e.dev, e.ctx.lib, e.ctx
        self.axy = torch.empty((n * k, 2), dtype=torch.float64, device=dev)
        self.bxy = torch.empty((n * k, 2), dtype=torch.float64, device=dev)
        self.aoff = torch.empty(n + 1, dtype=torch.int64, device=dev)
        self.boff = torch.empty(n + 1, dtype=torch.int64, device=dev)
        E.check(lib.gpl_gen_walk_linestrings(ctx._h, 3, -1, lo, n, k, self.axy.data_ptr(), self.aoff.data_ptr()))
        E.check(lib.gpl_gen_walk_linestrings(ctx._h, 4, 3, lo, n, k, self.bxy.data_ptr(), self.boff.data_ptr()))
        self.A = ctx.wrap_device(GeometryType.LINESTRING, n, n * k, self.axy.data_ptr(), geom_off_ptr=self.aoff.data_ptr(), keepalive=(self.axy, self.aoff))
        self.B = ctx.wrap_device(GeometryType.LINESTRING, n, n * k, self.bxy.data_ptr(), geom_off_ptr=self.boff.data_ptr(), keepalive=(self.bxy, self.boff))
        self.dist_out = torch.empty(n, dtype=torch.float64, device=dev)
        self.bits = torch.empty((n + 7) // 8, dtype=torch.uint8, device=dev)
        self.units_per_rank = n
        self.algo_bytes = 2 * n * k * COORD_BYTES * 2  # both kernels read both coordinate columns
        self.write_bytes = n * 8 + (n + 7) // 8

    def step(self, events):
        import torch

        from geopolars_b200 import engine as E

        e = self.env
        if events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(e.stream)
        E.check(e.ctx.lib.gpl_distance(e.ctx._h, self.A._h, self.B._h, C.c_void_p(self.dist_out.data_ptr()), None, E.GPL_DEVICE))
        E.check(e.ctx.lib.gpl_intersects(e.ctx._h, self.A._h, self.B._h, C.c_void_p(self.bits.data_ptr()), E.GPL_DEVICE))
        if events is not None:
            e1.record(e.stream)
            events.append((e0, e1))

    def describe_step(self):
        return "euclidean distance (f64 column) + intersects (bitmap) over this rank's row range; results stay row-partitioned (no collective)"

    def workload_text(self):
        return f"{self.total} LineString pairs, {self.K} coordinates each, euclidean_distance + intersects (BASELINE configs[2]; SURVEY.md config 3 generator)"

    def outputs(self):
        """distance and intersects (0 / 1) of sampled pairs of this rank's row range"""
        import torch

        rows = sample_rows(self.n, 2_000_000, self.env.dev)
        bits = self.bits[rows // 8].to(torch.int64)
        return {"rows": rows, "distance": self.dist_out[rows], "intersects": (bits >> (rows % 8)) & 1}

    def verify(self):
        from geopolars_b200 import GeoArrowArray, synth
        from oracle import oracle as og

        m, k = min(self.n, self.args.verify_rows), self.K
        ah, _ = synth.walk_linestrings(m, k, first=self.lo, stream=3)
        bh, _ = synth.walk_linestrings(m, k, first=self.lo, stream=4, other_of=3)
        assert np.array_equal(self.axy[: m * k].cpu().numpy(), ah) and np.array_equal(self.bxy[: m * k].cpu().numpy(), bh), "device RNG differs from the host RNG"
        off = np.arange(m + 1) * k
        HA = og.OGArray(og.LINESTRING, ah, geom_off=off)
        HB = og.OGArray(og.LINESTRING, bh, geom_off=off)
        th = len(all_cpus())
        want_i = og.intersects_rowwise(HA, HB, threads=th)
        want_d = og.distance_rowwise(HA, HB, threads=th)
        got_i = np.unpackbits(self.bits[: (m + 7) // 8].cpu().numpy(), bitorder="little")[:m].astype(bool)
        got_d = self.dist_out[:m].cpu().numpy()
        assert np.array_equal(got_i, want_i), "intersects differs from the oracle"
        denom = np.maximum(np.abs(want_d), np.abs(got_d))
        denom[denom == 0] = 1.0
        assert (np.abs(got_d - want_d) <= 1e-9 * denom).all(), "distance differs from the oracle by more than 1e-9 relative"
        assert np.array_equal(got_d == 0.0, want_i)
        return {"rows_checked_per_rank": m, "intersects_equal_oracle": True, "distance_within_1e-9": True, "intersecting_fraction": float(want_i.mean())}

    def e2e_setup(self):
        import torch

        n, k = self.n, self.K
        self.h_axy = torch.empty((n * k, 2), dtype=torch.float64, pin_memory=True)
        self.h_bxy = torch.empty((n * k, 2), dtype=torch.float64, pin_memory=True)
        self.h_axy.copy_(self.axy)
        self.h_bxy.copy_(self.bxy)
        self.h_off = (np.arange(n + 1, dtype=np.int64) * k)
        self.h_dist = torch.empty(n, dtype=torch.float64, pin_memory=True)
        self.h_bits = torch.empty((n + 7) // 8, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        self.h2d = 2 * (n * k * COORD_BYTES + (n + 1) * 8)
        self.d2h = n * 8 + (n + 7) // 8
        self.e2e_path = "gpl_array_from_buffers(host) x 2 + gpl_distance + gpl_intersects with host outputs"

    def e2e_step(self):
        from geopolars_b200 import GeoArrowArray
        from geopolars_b200 import engine as E

        ctx = self.env.ctx
        a = ctx.upload(GeoArrowArray.linestrings(self.h_axy.numpy(), self.h_off))
        b = ctx.upload(GeoArrowArray.linestrings(self.h_bxy.numpy(), self.h_off))
        E.check(ctx.lib.gpl_distance(ctx._h, a._h, b._h, C.c_void_p(self.h_dist.data_ptr()), None, E.GPL_HOST))
        E.check(ctx.lib.gpl_intersects(ctx._h, a._h, b._h, C.c_void_p(self.h_bits.data_ptr()), E.GPL_HOST))
        return (a, b)

    def e2e_check(self):
        import torch

        assert torch.equal(self.h_dist, self.dist_out.cpu()) and torch.equal(self.h_bits, self.bits.cpu()), "e2e results differ from the resident run"

    def cpu_sample(self, n_sample, threads):
        from geopolars_b200 import synth
        from oracle import oracle as og

        k = self.K
        ah, _ = synth.walk_linestrings(n_sample, k, stream=3)
        bh, _ = synth.walk_linestrings(n_sample, k, stream=4, other_of=3)
        off = np.arange(n_sample + 1) * k
        HA, HB = og.OGArray(og.LINESTRING, ah, geom_off=off), og.OGArray(og.LINESTRING, bh, geom_off=off)
        og.distance_rowwise(og.OGArray(og.LINESTRING, ah[: 1000 * k], geom_off=off[:1001]), og.OGArray(og.LINESTRING, bh[: 1000 * k], geom_off=off[:1001]), threads=threads)
        t0 = time.perf_counter()
        og.distance_rowwise(HA, HB, threads=threads)
        og.intersects_rowwise(HA, HB, threads=threads)
        dt = time.perf_counter() - t0
        return n_sample / dt, dt, f"{n_sample} of {self.total} pairs, distance + intersects, OpenMP static row chunks"

    def default_cpu_sample(self):
        return 2_000_000


class HullWorkload:
    """c5: convex_hull + affine_transform over 257-coordinate polygons (geoseries.rs:11-12, 23-26)"""

    NV = 256
    MATRIX = (0.8, -0.6, 10.0, 0.6, 0.8, -5.0)

    def __init__(self, name, args, env):
        self.name, self.args, self.env = name, args, env
        self.total = args.points or 10_000_000
        self.unit_name = "polygons"
        self.scaling = "strong"
        self.kernel = "k_hull_fast (+ k_hull on flagged rows; convex_hull) + k_affine (affine_transform)"
        self.traffic_file = "r2_hull_traffic.json"

    def setup(self):
        import torch

        from geopolars_b200 import GeometryType
        from geopolars_b200 import dist as gd
        from geopolars_b200 import engine as E

        e = self.env
        lo, hi = gd.shard_rows(self.total, e.world, e.rank)  # equal coordinate counts per row: row ranges are coordinate-balanced
        g, nv = hi - lo, self.NV
        self.lo, self.g = lo, g
        nc = g * (nv + 1)
        self.nc = nc
        self.xy = torch.empty((nc, 2), dtype=torch.float64, device=e.dev)
        self.ro = torch.empty(g + 1, dtype=torch.int64, device=e.dev)
        self.go = torch.empty(g + 1, dtype=torch.int64, device=e.dev)
        E.check(e.ctx.lib.gpl_gen_blob_polygons(e.ctx._h, 5, lo, g, nv, self.xy.data_ptr(), self.ro.data_ptr(), self.go.data_ptr()))
        self.polys = e.ctx.wrap_device(GeometryType.POLYGON, g, nc, self.xy.data_ptr(), geom_off_ptr=self.go.data_ptr(), ring_off_ptr=self.ro.data_ptr(),
                                       n_rings=g, keepalive=(self.xy, self.ro, self.go))
        self.hull = self.moved = None
        self.units_per_rank = g
        self.algo_bytes = 2 * nc * COORD_BYTES  # hull reads the coordinates once, affine once
        self.write_bytes = nc * COORD_BYTES  # + 16 h per hull ring, reported from the last step

    def step(self, events):
        import torch
        import torch.distributed as dist

        from geopolars_b200 import engine as E

        e = self.env
        self.hull = self.moved = None  # previous step's outputs go back to the context cache first
        if events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(e.stream)
        self.hull = E.convex_hull(self.polys)
        self.moved = E.affine_transform(self.polys, self.MATRIX)
        if events is not None:
            e1.record(e.stream)
            events.append((e0, e1))
        if e.world > 1:
            # ragged gather of the hull rings on rank 0: ring lengths (fixed width), then the coordinates (variable width)
            hv = self.hull.view()
            sizes = torch.empty(self.g + 1, dtype=torch.int64, device=e.dev)
            coords = torch.empty((hv.n_coords, 2), dtype=torch.float64, device=e.dev)
            E.check(e.ctx.lib.gpl_array_copy_out(e.ctx._h, self.hull._h, C.c_void_p(coords.data_ptr()), None, None, C.c_void_p(sizes.data_ptr()), None, E.GPL_DEVICE))
            g_max = (self.total + e.world - 1) // e.world + 1
            ring_off_pad = torch.zeros(g_max + 1, dtype=torch.int64, device=e.dev)
            ring_off_pad[: self.g + 1] = sizes  # this rank's ring offsets (rebased on rank 0 from the coordinate counts)
            self.gathered_ring_off = [torch.empty_like(ring_off_pad) for _ in range(e.world)] if e.rank == 0 else None
            dist.gather(ring_off_pad, self.gathered_ring_off, dst=0)
            ncoords = torch.tensor([hv.n_coords], dtype=torch.int64, device=e.dev)
            all_n = [torch.zeros(1, dtype=torch.int64, device=e.dev) for _ in range(e.world)]
            dist.all_gather(all_n, ncoords)
            counts = [int(t.item()) for t in all_n]
            if e.rank == 0:
                self.gathered = [coords] + [torch.empty((c, 2), dtype=torch.float64, device=e.dev) for c in counts[1:]]
                ops = [dist.P2POp(dist.irecv, self.gathered[r], r) for r in range(1, e.world)]
            else:
                ops = [dist.P2POp(dist.isend, coords, 0)]
            for w in dist.batch_isend_irecv(ops):
                w.wait()
            self.gather_bytes = sum(counts) * COORD_BYTES

    def describe_step(self):
        s = "convex_hull (variable-length rings: count/scan/write) + affine_transform over this rank's row range"
        if self.env.world > 1:
            s += " + ragged gather of the hull rings on rank 0 (all-gather of sizes, grouped send/recv of coordinates)"
        return s

    def workload_text(self):
        return f"{self.total} polygons x {self.NV + 1} coordinates, convex_hull + affine_transform (BASELINE configs[4]; SURVEY.md config 5 generator)"

    def hull_rings(self):
        """the last step's hull column as device tensors: ring offsets (g + 1) and coordinates"""
        import torch

        from geopolars_b200 import engine as E

        e = self.env
        hro = torch.empty(self.g + 1, dtype=torch.int64, device=e.dev)
        hxy = torch.empty((self.hull.view().n_coords, 2), dtype=torch.float64, device=e.dev)
        E.check(e.ctx.lib.gpl_array_copy_out(e.ctx._h, self.hull._h, C.c_void_p(hxy.data_ptr()), None, None, C.c_void_p(hro.data_ptr()), None, E.GPL_DEVICE))
        e.stream.synchronize()
        return hro, hxy

    def moved_coords(self):
        """the last step's affine_transform output as a (coordinates, 2) device tensor"""
        import torch

        from geopolars_b200 import engine as E

        e = self.env
        mv = torch.empty((self.nc, 2), dtype=torch.float64, device=e.dev)
        E.check(e.ctx.lib.gpl_array_copy_out(e.ctx._h, self.moved._h, C.c_void_p(mv.data_ptr()), None, None, None, None, E.GPL_DEVICE))
        e.stream.synchronize()
        return mv

    def outputs(self):
        """hull rings (coordinate counts and concatenated coordinates) and transformed coordinates of sampled polygons"""
        import torch

        rows = sample_rows(self.g, 4096, self.env.dev)
        hro, hxy = self.hull_rings()
        start = hro[rows]
        lens = hro[rows + 1] - start
        first = torch.cumsum(lens, 0) - lens  # where each sampled ring starts in the concatenation
        at = torch.repeat_interleave(start - first, lens) + torch.arange(int(lens.sum()), device=self.env.dev)
        moved = self.moved_coords().view(self.g, self.NV + 1, 2)[rows].reshape(-1, 2)
        return {"rows": rows, "hull_ring_len": lens, "hull_xy": hxy[at], "affine_xy": moved}

    def verify(self):
        from oracle import oracle as og

        m, nv = min(self.g, self.args.verify_rows), self.NV
        hv = self.hull.view()
        hro, hxy = self.hull_rings()
        xy = self.xy[: m * (nv + 1)].cpu().numpy()  # the device generator uses CUDA sincos: the oracle gets the device's coordinates
        ro = np.arange(m + 1, dtype=np.int64) * (nv + 1)
        arr = og.OGArray(og.POLYGON, xy, geom_off=np.arange(m + 1, dtype=np.int64), ring_off=ro)
        want_off, want_xy = og.convex_hull(arr, threads=len(all_cpus()))
        got_off = hro[: m + 1].cpu().numpy()
        assert np.array_equal(got_off, want_off), "hull ring offsets differ from the oracle"
        assert np.array_equal(hxy[: int(got_off[-1])].cpu().numpy(), want_xy), "hull rings differ from the oracle (vertex set or order)"
        mv = self.moved_coords()
        assert np.array_equal(mv[: m * (nv + 1)].cpu().numpy(), og.affine_transform(xy, self.MATRIX, threads=len(all_cpus()))), "affine_transform is not bit-exact"
        self.write_bytes = self.nc * COORD_BYTES + hv.n_coords * COORD_BYTES
        return {"rows_checked_per_rank": m, "hull_rings_bit_identical": True, "affine_bit_exact": True, "hull_mean_vertices": hv.n_coords / max(1, self.g)}

    def e2e_setup(self):
        import torch

        g = min(self.g, 1_000_000)  # host image of 1 M polygons (4.1 GB) — the full 41 GB column is not staged in host memory
        self.e2e_g = g
        nc = g * (self.NV + 1)
        self.h_xy = torch.empty((nc, 2), dtype=torch.float64, pin_memory=True)
        self.h_xy.copy_(self.xy[:nc])
        torch.cuda.synchronize()
        self.h_ro = np.arange(g + 1, dtype=np.int64) * (self.NV + 1)
        self.h_go = np.arange(g + 1, dtype=np.int64)
        self.h2d = nc * COORD_BYTES + 16 * (g + 1)
        self.d2h = nc * COORD_BYTES  # + hull rings, added after the first run
        self.e2e_units = g
        self.e2e_path = f"{g} polygons per rank per step: gpl_array_from_buffers(host) + gpl_convex_hull + gpl_affine_transform + gpl_array_copy_out(host) of both results"

    def e2e_step(self):
        from geopolars_b200 import GeoArrowArray
        from geopolars_b200 import engine as E

        ctx = self.env.ctx
        d = ctx.upload(GeoArrowArray.polygons(self.h_xy.numpy(), self.h_ro, self.h_go))
        h = E.convex_hull(d).to_host()
        a = E.affine_transform(d, self.MATRIX).to_host()
        self.d2h = a.xy.nbytes + h.xy.nbytes + h.ring_off.nbytes
        return (h, a)

    def e2e_check(self):
        pass

    def cpu_sample(self, n_sample, threads):
        from geopolars_b200 import synth
        from oracle import oracle as og

        xy, ro, go = synth.blob_polygons(n_sample, self.NV, stream=5)
        arr = og.OGArray(og.POLYGON, xy, geom_off=go, ring_off=ro)
        t0 = time.perf_counter()
        og.convex_hull(arr, threads=threads)
        og.affine_transform(xy, self.MATRIX, threads=threads)
        dt = time.perf_counter() - t0
        return n_sample / dt, dt, f"{n_sample} of {self.total} polygons, convex_hull + affine_transform, OpenMP static row chunks"

    def default_cpu_sample(self):
        return 400_000


WORKLOADS = {"c2": JoinWorkload, "c4": JoinWorkload, "c3": PairsWorkload, "c5": HullWorkload}


class Env:
    pass


def best_cpu_threads(wl, probe):
    """all logical CPUs or one per physical core, whichever runs the CPU arm faster on a small probe
    (the ring walk is latency bound; hyper-threads can hurt)"""
    cpus = len(all_cpus())
    best, best_rate = cpus, 0.0
    for th in sorted({cpus, max(1, cpus // 2)}, reverse=True):
        # best of two probes: under torchrun the sibling ranks are still starting up (and exiting) during the first one
        rate = max(wl.cpu_sample(probe, th)[0] for _ in range(2))
        if rate > best_rate:
            best, best_rate = th, rate
    return best


def cpu_arm_description():
    from oracle import oracle as og

    bi = og.build_info()
    return f"oracle/geo_oracle.c ({bi['flags']}) on {bi['cpu']}"


def run_reference(args, out):
    """--impl reference: the reference's CPU path (restated: oracle/geo_oracle.c, kind 'port') on the host cores."""
    if _env_int("RANK", 0) != 0:
        return 0
    env = Env()
    env.world, env.rank = max(1, args.gpus), 0
    wl = WORKLOADS[args.workload](args.workload, args, env)
    n_sample = args.ref_sample or 2 * wl.default_cpu_sample()
    threads = best_cpu_threads(wl, max(1, n_sample // 8))
    for _ in range(min(args.warmup, 2)):
        wl.cpu_sample(max(1, n_sample // 8), threads)
    times, desc = [], ""
    for _ in range(args.steps):
        _, dt, desc = wl.cpu_sample(n_sample, threads)
        times.append(dt)
    total_t = sum(times)
    value = n_sample * args.steps / total_t
    sample = f"{desc}; {cpu_arm_description()}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "geometries/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": wl.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.workload_text(),
                   "note": "reference arithmetic lives in un-vendored Rust crates (geo 0.27); this is the C restatement oracle/geo_oracle.c "
                           "timed on a bounded sample per step"},
        "cpu_baseline": {"value": value, "unit": "geometries/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "geometries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=out, flush=True)
    return 0


def main():
    # exactly ONE line goes to the real stdout (the JSON); anything libraries print (e.g. NCCL's version
    # banner when NCCL_DEBUG=VERSION) is sent to stderr instead
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    try:
        return _main(real_stdout)
    finally:
        real_stdout.flush()


def _main(out):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--points", type=int, default=0, help="units per GPU (c2/c4: points) or in total (c3: pairs, c5: polygons); 0 = the BASELINE size")
    ap.add_argument("--ref-sample", type=int, default=0, help="units per step of the CPU reference arm (0 = a default sized for ~10 s)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="units of the cpu_baseline sample (0 = default)")
    ap.add_argument("--verify-rows", type=int, default=10_000_000, help="rows per rank checked against the oracle after the timed region")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl b200")
    if args.workload in ("c3",):
        args.verify_rows = min(args.verify_rows, 2_000_000)
    if args.workload in ("c5",):
        args.verify_rows = min(args.verify_rows, 200_000)

    if args.impl == "reference":
        return run_reference(args, out)

    import torch
    import torch.distributed as dist

    from geopolars_b200 import engine as E

    env = Env()
    env.world = _env_int("WORLD_SIZE", 1)
    env.rank = _env_int("RANK", 0)
    local = _env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the geopolars_b200 path has no CPU fallback")
    torch.cuda.set_device(local)
    env.dev = torch.device("cuda", local)
    numa_node, full_affinity = (None, set(all_cpus()))
    if env.world > 1:
        numa_node, full_affinity = bind_to_gpu_numa_node(local)  # pinned host buffers on the GPU's socket
        dist.init_process_group("nccl", device_id=env.dev)
    warmup = max(args.warmup, 3)
    env.total_steps = warmup + args.steps
    env.stream = torch.cuda.Stream(device=env.dev)
    wl = WORKLOADS[args.workload](args.workload, args, env)
    with torch.cuda.stream(env.stream):
        env.ctx = E.Context(local, env.stream.cuda_stream)
        wl.setup()
        env.stream.synchronize()
        sampler = ClockSampler(local)
        if env.rank == 0:
            sampler.start()  # sampled from the warm-up on: the timed region alone can be shorter than one sample period
        t_load = time.perf_counter()
        for _ in range(warmup):
            wl.step(None)
        env.stream.synchronize()
        # nvidia-smi takes a few hundred ms to start and then reports every 20 ms, the default timed region lasts ~6 ms: keep
        # the device under the SAME load for MIN_LOAD_S before the timed region (more warm-up steps, in batches, the same
        # number on every rank) so that `clocks` holds samples taken under load right up to the timed steps.
        extra_warmup = 0
        while extra_warmup < 20000:
            go_on = 1 if time.perf_counter() - t_load < MIN_LOAD_S else 0
            if env.world > 1:
                flag = torch.tensor([go_on], dtype=torch.int32, device=env.dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
                go_on = int(flag.item())
            if not go_on:
                break
            for _ in range(8):
                wl.step(None)
            extra_warmup += 8
            env.stream.synchronize()
        if env.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        launches0 = env.ctx.launch_count
        env.ctx.kernel_timing(True)  # the library brackets each k_pip_stream launch with events on its stream
        events = []
        t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start.record(env.stream)
        for _ in range(args.steps):
            wl.step(events)
        t_end.record(env.stream)
        env.stream.synchronize()
        torch.cuda.synchronize()
        if env.world > 1:
            dist.barrier()
        launches = env.ctx.launch_count - launches0
        total_ms = t_start.elapsed_time(t_end)
        clocks = sampler.stop() if env.rank == 0 else None
        k_ms = [a.elapsed_time(b) for a, b in events]
        kt_ms, kt_n = env.ctx.kernel_timing_read()
        env.ctx.kernel_timing(False)
        # the dominant kernel alone when the library timed it (the join workloads), else the events around the op calls
        dom_ms = kt_ms / kt_n if kt_n else statistics.mean(k_ms)

        if args.dump_outputs and env.rank == 0:
            write_outputs(args.dump_outputs, wl.outputs())

        verify = None
        if not args.no_verify:
            verify = wl.verify()  # raises on any mismatch: an invalid number is not printed

        # ---- e2e: host buffers through the C ABI, copies inside the timed region --------------------
        e2e = None
        if not args.no_e2e:
            wl.e2e_setup()
            keep = None
            for _ in range(2):
                keep = wl.e2e_step()
            torch.cuda.synchronize()
            if env.world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                keep = wl.e2e_step()
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            wl.e2e_check()
            del keep
            e2e = {"seconds": e2e_s, "h2d": wl.h2d, "d2h": wl.d2h, "units": getattr(wl, "e2e_units", wl.units_per_rank)}

    # ---- reduce over ranks (max time) ------------------------------------------------------------------
    units_all = wl.units_per_rank
    if env.world > 1:
        t = torch.tensor([total_ms, e2e["seconds"] if e2e else 0.0, float(launches), float(statistics.mean(k_ms)), float(dom_ms)], dtype=torch.float64, device=env.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_max, launches, k_mean, dom_ms = t[0].item(), t[1].item(), int(t[2].item()), t[3].item(), t[4].item()
        if e2e:
            e2e["seconds"] = e2e_max
        u = torch.tensor([float(wl.units_per_rank), float(e2e["units"]) if e2e else 0.0], dtype=torch.float64, device=env.dev)
        dist.all_reduce(u)
        units_all = int(u[0].item())
        e2e_units_all = int(u[1].item())
    else:
        k_mean = statistics.mean(k_ms)
        e2e_units_all = e2e["units"] if e2e else 0
    if env.rank != 0:
        if env.world > 1:
            dist.destroy_process_group()
        return 0

    ms_per_step = total_ms / args.steps
    value = units_all / (ms_per_step * 1e-3)
    peak, peak_src = measured_peaks()
    achieved = wl.algo_bytes / (dom_ms * 1e-3) / 1e9
    traffic = recorded_traffic(wl.traffic_file)
    line = {
        "metric": METRIC, "value": value, "unit": "geometries/s", "n_gpus": env.world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {
            "workload": wl.workload_text(),
            "step": wl.describe_step(),
            "l2": "inputs exceed the 126 MB L2 (>= 1.6 GB per GPU per step); no flush needed",
            "parallelism": f"row-range partition over {env.world} GPU(s)" + (", polygon side replicated" if args.workload in ("c2", "c4") else ""),
            "kernel_ms": dom_ms,
            "op_call_ms": k_mean,
            "warmup_steps_run": warmup + extra_warmup,
            "timing": ("kernel_ms: CUDA events the library records around each k_pip_stream launch on its stream (gpl_ctx_kernel_timing); "
                       "op_call_ms: events around the whole gpl_contains_join call (counter memset + k_pip_stream + k_pip_deferred)"
                       if kt_n else "kernel_ms = op_call_ms: CUDA events around the op calls on the context's stream"),
            "numa_node": numa_node,
        },
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": (traffic or {}).get("dram_bytes_per_launch"), "traffic_source": (traffic or {}).get("source"),
                     "kernel": wl.kernel, "algorithmic_bytes_per_launch": wl.algo_bytes, "peak_source": peak_src,
                     "read_plus_write_GBps": (wl.algo_bytes + wl.write_bytes) / (dom_ms * 1e-3) / 1e9},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if verify is not None:
        line["verify"] = verify
    if e2e:
        line["e2e"] = {"value": e2e_units_all * args.steps / e2e["seconds"], "unit": "geometries/s", "h2d_bytes_per_step": e2e["h2d"],
                       "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": 1e3 * e2e["seconds"] / args.steps, "path": wl.e2e_path}
    if not args.no_cpu:
        if hasattr(os, "sched_setaffinity"):
            os.sched_setaffinity(0, full_affinity)  # the CPU arm gets every core again (this rank was bound to one socket)
        n_sample = args.cpu_sample or wl.default_cpu_sample()
        threads = best_cpu_threads(wl, max(1, n_sample // 8))
        v, dt, desc = wl.cpu_sample(n_sample, threads)
        line["cpu_baseline"] = {"value": v, "unit": "geometries/s", "cores": threads, "kind": "port",
                                "sample": f"{desc} in {dt:.2f} s; {cpu_arm_description()}"}
    print(json.dumps(line), file=out, flush=True)
    if env.world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
