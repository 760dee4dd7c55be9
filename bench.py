#!/usr/bin/env python
"""bench.py - front-end frames/s (+ local-BA solves/s) on N B200s vs the CPU reference path.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON
line on rank 0.  A "step" is one pass of the front-end hot path over one batch of B synthetic
(prev, cur) 640x480 frame pairs per GPU (BASELINE.json configs[1]):

    P  pyramids of prev and cur            (visual_front_end.cpp:1172)
    K  forward/backward KLT, 1024 kps/frame (feature_tracker.cpp:35-137; 60 % with a motion prior
       at nbpyrlvl 1, the rest at nbpyrlvl 3, as visual_front_end.cpp:196,242)
    F  detectGridFAST + cornerSubPix on cur (feature_extractor.cpp:443-570), parameters_files/fast:
       cell 50, nfast_th 10, no existing keypoints (full-grid detection)
    B  describeBRIEF of the tracked and of the new keypoints (feature_extractor.cpp:224-285)

  value  = frames/s with all inputs already resident in HBM (device pointers through the C ABI)
  e2e    = frames/s through the same C ABI calls with HOST (pinned) buffers: H2D of the images and
           keypoints and D2H of every result inside the timed region
  --impl reference : the reference's own CPU path (OpenCV call sequence, oracle/image_ref.py) on
           the box's host cores.

No part of the GPU arm touches oracle/; only the cpu_baseline leg and --impl reference do.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

W_IMG, H_IMG = 640, 480
NKP = 1024
CELL = 50
FAST_TH = 10
FRAC3D = 0.6


# ----------------------------------------------------------------------------- helpers
def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def usable_cores() -> int:
    """Host threads this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = max(1, min(n, int(float(q[0]) / float(q[1]) + 0.5)))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = max(1, min(n, int(quota / period + 0.5)))
        except Exception:
            pass
    return n


def _parse_cpulist(txt: str):
    out = []
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        out.extend(range(int(a), int(b or a) + 1))
    return out


def pin_to_gpu_numa(torch, local: int, world: int) -> dict:
    """Multi-rank runs: bind this rank (and the chunk threads / pinned buffers it creates afterwards: first touch) to
    the CPUs of the NUMA node its GPU hangs off, split evenly between the ranks of that node.  Round 1's 8-GPU e2e
    efficiency was 0.62 with every rank's threads and pinned pages floating over both sockets."""
    info = {"pinned": False}
    try:
        if world <= 1 or not hasattr(os, "sched_setaffinity"):
            return info
        allowed = sorted(os.sched_getaffinity(0))

        def node_cpus(dev):
            pr = torch.cuda.get_device_properties(dev)
            bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            txt = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read()
            return tuple(c for c in _parse_cpulist(txt) if c in allowed)

        mine = node_cpus(local)
        if not mine:
            return info
        ndev = min(world, torch.cuda.device_count())
        same = [d for d in range(ndev) if node_cpus(d) == mine]          # ranks sharing this NUMA node
        k, n = same.index(local), len(same)
        per = max(1, len(mine) // n)
        share = list(mine[k * per:(k + 1) * per]) or list(mine)
        os.sched_setaffinity(0, share)
        info = {"pinned": True, "cpus": len(share), "node_cpus": len(mine), "ranks_on_node": n}
    except Exception as e:      # pinning is an optimisation, never a failure
        info = {"pinned": False, "why": str(e)[:80]}
    return info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(", ") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows if len(r) >= 9]
            if sm:
                busy = [s for s in sm if s > 0.5 * max(sm)] or sm
                out["sm_mhz"] = float(np.median(busy))
                out["sm_max_mhz"] = float(rows[0][2])
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for k, nm in enumerate(names):
                    if any(r[5 + k].strip().lower().startswith("active") for r in rows if len(r) >= 9):
                        out["reasons"].append(nm)
            os.unlink(self.path)
        except Exception:
            pass
        return out


# ----------------------------------------------------------------------------- CPU reference arm
def _cpu_worker(args):
    """One worker: run the reference's OpenCV call sequence on a share of the frame pairs."""
    seeds, nkp = args
    import cv2
    cv2.setNumThreads(1)
    from oracle import image_ref as R
    from ov2slam_b200 import synth
    data = []
    for s in seeds:
        prev, cur, flow = synth.make_pair(s, W_IMG, H_IMG)
        rng = np.random.default_rng(s + 5)
        kps = np.stack([rng.uniform(12, W_IMG - 12, nkp), rng.uniform(12, H_IMG - 12, nkp)], axis=1).astype(np.float32)
        is3d, pri = synth.make_priors(s, kps, flow, FRAC3D)
        data.append((prev, cur, kps, pri, is3d))
    if data:  # untimed warm-up of this process (cv2 paging, detector creation)
        _cpu_frame(R, cv2, *data[0])
    t0 = time.perf_counter()
    ntracked = 0
    for prev, cur, kps, pri, is3d in data:
        r = _cpu_frame(R, cv2, prev, cur, kps, pri, is3d)
        ntracked += int(r)
    return time.perf_counter() - t0, len(data), ntracked


def _cpu_frame(R, cv2, prev, cur, kps, pri, is3d):
    """Same work as one GPU-arm frame: P(prev), P(cur), K (two calls), F + S (empty vcurkps), B.
    The Python binding of calcOpticalFlowPyrLK cannot take a prebuilt pyramid, so every LK call builds the
    pyramids it needs internally (2 per forward call; the reference builds each image's pyramid ONCE,
    visual_front_end.cpp:1172): no explicit buildOpticalFlowPyramid on top of that - the arm already does
    about twice the reference's pyramid work (~0.9 ms of ~12 ms per frame on one core)."""
    tracked = pri.copy()
    status = np.zeros(len(kps), np.uint8)
    i3 = np.nonzero(is3d)[0]
    i2 = np.nonzero(~is3d)[0]
    if len(i3):
        tracked[i3], status[i3] = R.fb_klt_cv2(prev, cur, kps[i3], tracked[i3], 9, 1)
    if len(i2):
        tracked[i2], status[i2] = R.fb_klt_cv2(prev, cur, kps[i2], tracked[i2], 9, 3)
    newpts, _, _ = R.detect_grid_fast_cv2(cur, CELL, np.zeros((0, 2), np.float32), FAST_TH)
    R.describe_cv2(cur, tracked)
    R.describe_cv2(cur, newpts)
    return status.sum()


def run_cpu_reference(nframes: int, nproc: int, first_seed: int = 1000):
    """frames/s of the OpenCV reference sequence over `nframes` pairs with `nproc` processes.
    Input generation is outside the timed region (each worker times only its processing loop);
    throughput = frames / max worker time (workers run concurrently)."""
    import multiprocessing as mp
    nproc = max(1, min(nproc, nframes))
    seeds = [first_seed + i for i in range(nframes)]
    shares = [seeds[i::nproc] for i in range(nproc)]
    if nproc == 1:
        res = [_cpu_worker((shares[0], NKP))]
    else:
        ctxmp = mp.get_context("fork")
        with ctxmp.Pool(nproc) as pool:
            res = pool.map(_cpu_worker, [(s, NKP) for s in shares])
    tmax = max(r[0] for r in res)
    n = sum(r[1] for r in res)
    return n / tmax, tmax, n


def cpu_sample_frames(cores: int) -> int:
    """frame pairs per CPU-arm step: 32 per worker process (6 per worker gave +-40 % run to run), capped."""
    return int(min(max(32 * cores, 64), 3072))


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = usable_cores()
    nframes = cpu_sample_frames(cores)
    # warm-up steps (page in cv2, fork pool once) then K timed steps, each a bounded sample
    for _ in range(max(1, min(args.warmup, 1))):
        run_cpu_reference(min(nframes, cores), cores)
    vals = []
    t_total = 0.0
    for _ in range(args.steps):
        fps, t, n = run_cpu_reference(nframes, cores)
        vals.append(fps)
        t_total += t
    fps = float(np.mean(vals))
    try:
        import cv2
        ver = cv2.__version__
    except Exception:
        ver = "?"
    line = {
        "impl": "reference", "metric": "front-end frames/sec", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * t_total / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/i32/f32", "data": "synthetic",
        "config": _config(args.batch, "reference CPU arm: one step = a bounded sample of %d frame pairs of the same workload "
                                      "(frames/s is per frame, independent of the sample size)" % nframes),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{nframes} frame pairs/step, OpenCV {ver} call sequence of feature_tracker.cpp/"
                                   f"feature_extractor.cpp via cv2 (oracle/image_ref.py), {cores} processes x 1 cv2 thread"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def _config(batch, note=""):
    return {"workload": "C2: FAST+descriptor+fb-KLT front-end, batch of %d synthetic 640x480 frame pairs per GPU" % batch,
            "width": W_IMG, "height": H_IMG, "keypoints_per_frame": NKP, "klt": "win 9, nbpyrlvl 1 (60% prior) / 3, 30 it, eps 0.01, fb 0.5",
            "fast": "cell %d, th %d, full grid (no existing kps), cornerSubPix" % (CELL, FAST_TH),
            "descriptor": "ORB-fallback 256-bit (reference's non-contrib branch), tracked + new keypoints",
            "l2": "inputs (2 x batch x 307 KB = 157 MB at batch 256) exceed the 126 MB L2", "note": note}


# ----------------------------------------------------------------------------- GPU arm
class Workload:
    def __init__(self, torch, api, ctx, rank: int, batch: int):
        from ov2slam_b200 import synth
        self.torch, self.api, self.ctx, self.B = torch, api, ctx, batch
        dev = torch.device("cuda", torch.cuda.current_device())
        base = 1000 + rank * 100003
        prevs = np.empty((batch, H_IMG, W_IMG), np.uint8)
        curs = np.empty_like(prevs)
        kps = np.empty((batch, NKP, 2), np.float32)
        pri = np.empty_like(kps)
        lv = np.empty((batch, NKP), np.uint8)
        for i in range(batch):
            prevs[i], curs[i], flow = synth.make_pair(base + i, W_IMG, H_IMG)
            rng = np.random.default_rng(base + i + 5)
            kps[i] = np.stack([rng.uniform(12, W_IMG - 12, NKP), rng.uniform(12, H_IMG - 12, NKP)], axis=1)
            is3d, pri[i] = synth.make_priors(base + i, kps[i], flow, FRAC3D)
            lv[i] = np.where(is3d, 1, 3)
        self.ncell = (H_IMG // CELL) * (W_IMG // CELL)
        pin = lambda a: torch.from_numpy(a).pin_memory()
        # host (pinned) copies: the e2e arm reads inputs from and writes results to these
        self.h_prev, self.h_cur = pin(prevs), pin(curs)
        self.h_kps, self.h_pri0, self.h_lv = pin(kps.reshape(-1, 2)), pin(pri.reshape(-1, 2)), pin(lv.reshape(-1))
        n = batch * NKP
        self.h_pri = torch.empty((n, 2), dtype=torch.float32).pin_memory()
        self.h_status = torch.empty(n, dtype=torch.uint8).pin_memory()
        self.h_th = torch.empty(batch, dtype=torch.int32).pin_memory()
        self.h_new = torch.empty((batch * self.ncell, 2), dtype=torch.float32).pin_memory()
        self.h_cnt = torch.empty(batch, dtype=torch.int32).pin_memory()
        self.h_desc_t = torch.empty((n, 32), dtype=torch.uint8).pin_memory()
        self.h_val_t = torch.empty(n, dtype=torch.uint8).pin_memory()
        self.h_desc_n = torch.empty((batch * self.ncell, 32), dtype=torch.uint8).pin_memory()
        self.h_val_n = torch.empty(batch * self.ncell, dtype=torch.uint8).pin_memory()
        # device-resident copies for the `value` arm
        self.d_prev, self.d_cur = self.h_prev.to(dev), self.h_cur.to(dev)
        self.d_kps, self.d_pri0, self.d_lv = self.h_kps.to(dev), self.h_pri0.to(dev), self.h_lv.to(dev)
        self.d_pri = torch.empty_like(self.d_pri0)
        self.d_status = torch.empty(n, dtype=torch.uint8, device=dev)
        self.d_th = torch.empty(batch, dtype=torch.int32, device=dev)
        self.d_new = torch.empty((batch * self.ncell, 2), dtype=torch.float32, device=dev)
        self.d_cnt = torch.empty(batch, dtype=torch.int32, device=dev)
        self.d_desc_t = torch.empty((n, 32), dtype=torch.uint8, device=dev)
        self.d_val_t = torch.empty(n, dtype=torch.uint8, device=dev)
        self.d_desc_n = torch.empty((batch * self.ncell, 32), dtype=torch.uint8, device=dev)
        self.d_val_n = torch.empty(batch * self.ncell, dtype=torch.uint8, device=dev)
        # two pyramid sets: one aliasing the device images, one owning level 0 (host uploads)
        self.pyr_prev_d = api.Pyramid(ctx, batch, W_IMG, H_IMG, 3)
        self.pyr_cur_d = api.Pyramid(ctx, batch, W_IMG, H_IMG, 3)
        self.pyr_prev_h = api.Pyramid(ctx, batch, W_IMG, H_IMG, 3)
        self.pyr_cur_h = api.Pyramid(ctx, batch, W_IMG, H_IMG, 3)
        self.ft = api.FeatureTracker(ctx, 30, 0.01)
        self.fe = api.FeatureExtractor(ctx, nmaxdist=CELL, nfast_th=FAST_TH)
        self.h2d = (self.h_prev.numel() + self.h_cur.numel() + self.h_kps.numel() * 4 + self.h_pri0.numel() * 4 +
                    self.h_lv.numel() + self.h_th.numel() * 4 + n * 8 + batch * self.ncell * 8)
        self.d2h = (n * 8 + n + batch * 4 + batch * self.ncell * 8 + batch * 4 + n * 33 + batch * self.ncell * 33)

    def step_resident(self):
        B, n = self.B, self.B * NKP
        self.pyr_prev_d.build(self.d_prev)
        self.pyr_cur_d.build(self.d_cur)
        self.d_pri.copy_(self.d_pri0)          # vpriorkps is in/out: fresh guess every step
        self.d_th.fill_(FAST_TH)               # constant work per step
        self.ft.fb_klt_tracking(self.pyr_prev_d, self.pyr_cur_d, 9, self.d_lv, 30.0, 0.5, self.d_kps, self.d_pri,
                                self.d_status, n=n, per_frame=NKP)
        self.fe.detect_grid_fast(self.pyr_cur_d, CELL, 0, B, self.d_th, self.d_new, self.d_cnt, max_per_frame=self.ncell)
        self.fe.describe_brief(self.pyr_cur_d, self.d_pri, self.d_desc_t, self.d_val_t, n=n, per_frame=NKP)
        self.fe.describe_brief(self.pyr_cur_d, self.d_new, self.d_desc_n, self.d_val_n, n=B * self.ncell, per_frame=self.ncell)

    def dump_outputs(self, out_dir: str, max_bytes: int = 64 << 20):
        """Write what the last resident step computed, frame by frame, as float32 DIR/<name>.npy: the tracked keypoints and
        their status, the adapted FAST thresholds, the new keypoints and their count, and the descriptors of both with their
        validity flags.  Slots past a frame's new-keypoint count and descriptors flagged invalid hold no result and are written
        as 0.  A batch whose outputs exceed `max_bytes` is written for a fixed, seeded sample of its frames (frame_index.npy)."""
        self.torch.cuda.synchronize()
        B, nc = self.B, self.ncell
        get = lambda t, *shape: t.cpu().numpy().reshape(B, *shape)
        out = {"tracked_kps": get(self.d_pri, NKP, 2), "track_status": get(self.d_status, NKP), "fast_threshold": get(self.d_th),
               "new_kps": get(self.d_new, nc, 2), "new_count": get(self.d_cnt), "tracked_desc": get(self.d_desc_t, NKP, 32),
               "tracked_desc_valid": get(self.d_val_t, NKP), "new_desc": get(self.d_desc_n, nc, 32), "new_desc_valid": get(self.d_val_n, nc)}
        empty = np.arange(nc)[None, :] >= out["new_count"][:, None]
        out["new_kps"][empty] = 0
        out["new_desc_valid"][empty] = 0
        out["tracked_desc"][out["tracked_desc_valid"] == 0] = 0
        out["new_desc"][out["new_desc_valid"] == 0] = 0
        frame_bytes = 4 * (1 + sum(a[0].size for a in out.values()))
        frames = np.arange(B)
        if B * frame_bytes > max_bytes:
            frames = np.sort(np.random.default_rng(0).choice(B, max_bytes // frame_bytes, replace=False))
        out = {k: v[frames] for k, v in out.items()}
        out["frame_index"] = frames
        os.makedirs(out_dir, exist_ok=True)
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v.astype(np.float32))

    # ---- end-to-end arm: the batch is cut into chunks, each chunk goes through the same C-ABI calls
    # with HOST pointers on its own context (= its own stream) from its own host thread, so the
    # H2D/D2H copies of one chunk overlap the kernels of another (the reference itself runs its
    # front-end and mapper in separate threads; one ov2_ctx per thread is the documented usage).
    def init_e2e(self, nchunks: int):
        import concurrent.futures as cf
        api, torch = self.api, self.torch
        self.nchunks = nchunks
        self.cs = self.B // nchunks
        assert self.cs * nchunks == self.B
        self.ectx, self.epp, self.ecp, self.eft, self.efe = [], [], [], [], []
        for k in range(nchunks):
            c = api.Context(torch.cuda.current_device())
            self.ectx.append(c)
            self.epp.append(api.Pyramid(c, self.cs, W_IMG, H_IMG, 3))
            self.ecp.append(api.Pyramid(c, self.cs, W_IMG, H_IMG, 3))
            self.eft.append(api.FeatureTracker(c, 30, 0.01))
            self.efe.append(api.FeatureExtractor(c, nmaxdist=CELL, nfast_th=FAST_TH))
        self.pool = cf.ThreadPoolExecutor(max_workers=nchunks)
        self._e2e_prepare()

    def _e2e_prepare(self):
        """Per-chunk raw host addresses, computed once: the timed loop then only makes ctypes calls
        (which release the GIL) - no numpy/torch view construction under the GIL per step."""
        self._cargs = []
        for k in range(self.nchunks):
            cs, nk, nc = self.cs, self.cs * NKP, self.cs * self.ncell
            f0, k0, c0 = k * cs, k * cs * NKP, k * cs * self.ncell
            adr = lambda t, a: t[a:a + 1].data_ptr() if t.numel() else 0
            self._cargs.append(dict(
                prev=adr(self.h_prev, f0), cur=adr(self.h_cur, f0), lv=adr(self.h_lv, k0), kps=adr(self.h_kps, k0),
                pri=adr(self.h_pri, k0), pri0=adr(self.h_pri0, k0), status=adr(self.h_status, k0), th=adr(self.h_th, f0),
                new=adr(self.h_new, c0), cnt=adr(self.h_cnt, f0), desc_t=adr(self.h_desc_t, k0), val_t=adr(self.h_val_t, k0),
                desc_n=adr(self.h_desc_n, c0), val_n=adr(self.h_val_n, c0), nk=nk, nc=nc, cs=cs,
                th_view=self.h_th[f0:f0 + cs], pri_view=self.h_pri[k0:k0 + nk], pri0_view=self.h_pri0[k0:k0 + nk]))
            c = self._cargs[-1]
            c["step_args"] = self.api.FrontendStepArgs(
                c["prev"], c["cur"], W_IMG, W_IMG * H_IMG, cs, self.api.KltParams(9, 30, float(np.float32(0.01)), 30.0, 0.5),
                nk, NKP, c["lv"], 0, c["kps"], c["pri"], c["status"], CELL, c["th"], self.ncell, c["new"], c["cnt"],
                c["desc_t"], c["val_t"], c["desc_n"], c["val_n"])

    def _e2e_chunk(self, k: int):
        a = self._cargs[k]
        pp, cp, ft, fe = self.epp[k], self.ecp[k], self.eft[k], self.efe[k]
        a["pri_view"].copy_(a["pri0_view"])         # vpriorkps is in/out: fresh guess every step
        a["th_view"].fill_(FAST_TH)
        self.api.frontend_step(self.ectx[k], pp, cp, a["step_args"])   # one ABI call: H2D, kernels, D2H, one sync

    def step_e2e(self):
        list(self.pool.map(self._e2e_chunk, range(self.nchunks)))
        return int(self.h_cnt.sum())          # the step's result is read on the host (new keypoint counts)

    def _e2e_chunk_stream(self, k: int, steps: int):
        a = self._cargs[k]
        f0, cs = k * self.cs, self.cs
        total = 0
        for _ in range(steps):
            self._e2e_chunk(k)
            total += int(self.h_cnt[f0:f0 + cs].sum())   # this chunk's result of this step, read on the host
        return total

    def stream_e2e(self, steps: int):
        """`steps` steps, pipelined: every chunk thread runs its share of each step back to back, so the
        uploads of step s+1 overlap the kernels of step s (a streaming front-end; no barrier between
        steps).  Every step still uploads all its inputs and reads all its results on the host."""
        return sum(self.pool.map(lambda k: self._e2e_chunk_stream(k, steps), range(self.nchunks)))

    def e2e_launches(self):
        return sum(c.launch_count() for c in self.ectx)

    def close(self):
        if hasattr(self, "pool"):
            self.pool.shutdown(wait=True)
        for p in getattr(self, "epp", []) + getattr(self, "ecp", []) + [self.pyr_prev_d, self.pyr_cur_d, self.pyr_prev_h, self.pyr_cur_h]:
            p.close()
        for c in getattr(self, "ectx", []):
            c.close()


# SURVEY.md 8(d) algorithmic bytes per unit (stated in DESIGN.md)
def algorithmic_bytes(kernel: str, batch: int) -> float:
    wh = W_IMG * H_IMG
    ncell = (H_IMG // CELL) * (W_IMG // CELL)
    if kernel == "fb_klt_kernel":       # per keypoint: fwd 0.9 KB + bwd 0.22 KB compulsory gathers
        return batch * NKP * (900.0 + 220.0)
    if kernel == "pyr_down_kernel":     # per frame and level pair: read level, write quarter (3 launches / pyramid)
        return batch * wh * (1 + 0.25 + 0.25 + 0.0625 + 0.0625 + 0.015625) / 3.0
    if kernel == "fast_cells_kernel":   # read the cells once + candidate lists
        return batch * (ncell * CELL * CELL + ncell * 8.0)
    if kernel == "fast_sweep_kernel":
        return batch * ncell * 64.0
    if kernel == "subpix_kernel":
        return batch * ncell * (81.0 * 4 + 16)
    if kernel == "describe_kernel":     # 32x32 raw window + 32 B descriptor per keypoint
        return batch * NKP * (1024.0 + 40.0)
    return 0.0


def gpu_arm(args):
    import torch
    import torch.distributed as dist
    from ov2slam_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback")
    torch.cuda.set_device(local)
    numa = pin_to_gpu_numa(torch, local, world)      # before any pinned allocation / thread pool (first touch)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # a real (non-default) stream: the C ABI context launches on it and torch's helper ops
    # (copy_/fill_) are ordered with the kernels because it is also torch's current stream
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = api.Context(local, stream=stream.cuda_stream)
    if args.kernels_only and args.only in ("c4", "c5"):
        # profiler runs of the other legs: resident steps only (no host threads under ncu)
        import bench_legs as L
        if args.only == "c4":
            w4 = L.C4Workload(torch, api, ctx, rank, args.c4_batch, args.c4_unique, min(usable_cores(), 16))
            for _ in range(args.warmup + args.steps):
                w4.step_resident()
            torch.cuda.synchronize()
        else:
            from ov2slam_b200 import synth
            pb = synth.make_ba_problem(5, *(L.C5 if not args.c5_small else (20, 3000, 18000)))
            opt = api.Optimizer(ctx)
            for _ in range(args.warmup + args.steps):
                opt.local_ba({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()})
        print(json.dumps({"kernels_only": True, "only": args.only, "note": "not a bench line: for ncu"}), flush=True)
        return 0
    wl = Workload(torch, api, ctx, rank, args.batch)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        launches = ctx.launch_count() - l0
        t = torch.tensor([ms, wall * 1000.0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), launches

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_res, wall_res, launches = timed(wl.step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        wl.dump_outputs(args.dump_outputs)
    if args.kernels_only:
        # profiler runs (ncu serialises kernels; the multi-threaded e2e arm must not run under it)
        if rank == 0:
            sampler.stop()
            print(json.dumps({"kernels_only": True, "ms_per_step": ms_res / args.steps, "batch": args.batch,
                              "note": "not a bench line: resident steps only, for ncu"}), flush=True)
        return 0
    if args.e2e_chunks <= 0:
        args.e2e_chunks = 8 if world == 1 else max(4, min(8, usable_cores()))
    while args.batch % args.e2e_chunks:
        args.e2e_chunks -= 1
    wl.init_e2e(args.e2e_chunks)
    ms_e2e_dev, wall_e2e, _ = timed(wl.step_e2e, args.steps, max(1, args.warmup))
    # device events miss host-side staging of the last D2H sync; use the larger of event/wall time for e2e
    ms_e2e_stepped = max(ms_e2e_dev, wall_e2e)
    # pipelined variant (the headline e2e): same K steps, same copies, no barrier between steps.
    # The K-step region is timed three times and the MEDIAN is reported (host-thread scheduling on the
    # box's CPU quota makes single regions of ~0.1 s noisy); all three are kept in the JSON line.
    wl.stream_e2e(max(1, args.warmup))
    stream_ms = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        wl.stream_e2e(args.steps)
        torch.cuda.synchronize()
        tp = torch.tensor([(time.perf_counter() - t0) * 1000.0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        stream_ms.append(float(tp[0]))
    ms_e2e_stream = sorted(stream_ms)[1]
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e = ms_e2e_stepped if args.e2e_stepped else ms_e2e_stream
    frames = world * args.batch * args.steps
    value = frames / (ms_res / 1000.0)
    e2e = frames / (ms_e2e / 1000.0)

    line = None
    if rank == 0:
        # roofline pass: per-kernel CUDA-event durations on the launching stream (separate, untimed run)
        ctx.profile(True)
        for _ in range(3):
            wl.step_resident()
        rep = ctx.profile_report()
        ctx.profile(False)
        peak, peak_src = _peaks()
        tot = sum(v[0] for v in rep.values()) or 1.0
        dom = max(rep.items(), key=lambda kv: kv[1][0])
        dname, (dms, dn) = dom
        avg_ms = dms / dn
        alg = algorithmic_bytes(dname, args.batch)
        if dname == "describe_kernel":   # two launches of different size per step: use the per-step total
            alg = args.batch * (NKP + (H_IMG // CELL) * (W_IMG // CELL)) * 1064.0 / 2.0
        achieved = alg / (avg_ms * 1e-3) / 1e9
        shares = {k: round(v[0] / tot, 4) for k, v in rep.items()}
        roof = {"bound": "hbm", "kernel": dname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": _ncu_traffic(dname), "peak_source": peak_src,
                "avg_launch_ms": avg_ms, "algorithmic_bytes_per_launch": alg, "kernel_time_shares": shares,
                "note": "KLT is gather/iteration bound by construction (SURVEY.md 8d-ii): HBM fraction is low by design"}
        cores = usable_cores()
        cpu = None
        if world == 1 and not args.no_cpu:
            nfr = cpu_sample_frames(cores)
            fps, t, n = run_cpu_reference(nfr, cores)
            fps1, t1, n1 = run_cpu_reference(16, 1)
            try:
                import cv2
                ver = cv2.__version__
            except Exception:
                ver = "?"
            try:
                simd = [l.strip() for l in cv2.getBuildInformation().splitlines() if "CPU/HW features" in l or "Baseline:" in l or "Dispatched" in l][:3]
            except Exception:
                simd = []
            cpu = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "single_core_value": fps1,
                   "sample": f"{n} frame pairs, OpenCV {ver} call sequence (oracle/image_ref.py) in {cores} processes x 1 cv2 thread; "
                             f"single core: {fps1:.1f} frames/s on {n1} pairs; LK rebuilds its pyramids per call (about 2x the "
                             f"reference's pyramid work)", "opencv_simd": simd}
        line = {
            "metric": "front-end frames/sec", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/i32/f32",
            "data": "synthetic", "config": _config(args.batch, "per-GPU batch fixed (weak scaling); no data-path collective"),
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(wl.h2d), "d2h_bytes_per_step": int(wl.d2h),
                    "ms_per_step": ms_e2e / args.steps, "chunks": args.e2e_chunks, "numa": numa,
                    "mode": "stepped (barrier after every step)" if args.e2e_stepped else
                            "pipelined (chunk threads stream through the K steps; every step uploads its inputs and reads its results)",
                    "stepped_value": frames / (ms_e2e_stepped / 1000.0), "pipelined_value": frames / (ms_e2e_stream / 1000.0),
                    "pipelined_repeats": [frames / (m / 1000.0) for m in stream_ms]},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        }
    # free the C2 workload before the other legs allocate theirs
    wl.close()
    del wl
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    # ---- C4 (stereo 1280x720, accurate parameters) and C5 (localBA 150k observations, N-way) legs: every rank takes part
    import bench_legs as L
    legs = {}
    if not args.no_c4:
        try:
            legs["c4"] = L.c4_leg(torch, api, dist, ctx, stream, rank, world, args, _peaks(), usable_cores, _ncu_traffic)
        except Exception as e:  # a leg must never take the front-end line down
            import traceback
            legs["c4"] = {"error": (str(e) + " | " + traceback.format_exc().splitlines()[-2])[:400]}
    if not args.no_c5:
        try:
            legs["c5"] = L.c5_leg(torch, api, dist, ctx, rank, world, args, _peaks(), _ncu_traffic)
        except Exception as e:
            import traceback
            legs["c5"] = {"error": (str(e) + " | " + traceback.format_exc().splitlines()[-2])[:400]}
    if rank == 0:
        line.update(legs)
        if world == 1 and not args.no_ba:
            try:
                line["localba"] = ba_bench(torch, api, ctx)
            except Exception as e:
                line["localba"] = {"error": str(e)[:200]}
        if world == 1 and not args.no_cpu:
            try:
                line["class_path"] = class_path_bench()
            except Exception as e:
                line["class_path"] = {"error": str(e)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _ncu_traffic(kernel: str):
    """dram bytes per launch from the committed ncu summary (profiles/), or None."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    try:
        return json.loads(p.read_text()).get(kernel)
    except Exception:
        return None


def ba_bench(torch, api, ctx):
    """local-BA solves/s on the C3 problem (10 KF x 2000 pts x 8000 obs) - the second half of BASELINE.json's metric -
    through the C ABI with HOST buffers (upload of the flattened window, two-stage solve, download of poses / inverse
    depths / outlier flags all inside the timed region): one window per call (`value`) and K independent windows per
    launch (`batched`), next to the single-threaded C restatement of the reference's Ceres path (oracle/ba_ref_c.c;
    "restatement, not Ceres": Ceres cannot be built offline; the reference runs it with num_threads = 1,
    optimizer.cpp:460)."""
    from ov2slam_b200 import synth
    import bench_legs as L
    opt = api.Optimizer(ctx)
    pb0 = synth.make_ba_problem(3, 10, 2000, 8000)
    clone = lambda d=pb0: {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    reps, its = 50, 0
    for _ in range(3):
        opt.local_ba(clone())
    pbs = [clone() for _ in range(reps)]
    torch.cuda.synchronize()
    l0 = ctx.launch_count()
    t0 = time.perf_counter()
    for pb in pbs:
        res, _ = opt.local_ba(pb)
        its += res["iters_robust"] + res["iters_refine"]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    launches = (ctx.launch_count() - l0) / reps
    ctx.profile(True)
    opt.local_ba(clone())
    rep = ctx.profile_report()
    ctx.profile(False)
    tot = sum(v[0] for v in rep.values()) or 1.0
    peak, peak_src = _peaks()
    bpi = L.ba_bytes_per_iteration(8000, 2000)
    out = {"metric": "local-BA solves/sec", "value": reps / dt, "unit": "solves/s", "ms_per_solve": 1e3 * dt / reps,
           "config": {"workload": "C3: localBA 10 KF x 2000 inverse-depth pts x 8000 obs, 5 % gross outliers, two-stage solve"},
           "lm_iterations_per_solve": its / reps, "final_cost": res["final_cost"], "dtype": "f64",
           "kernel_time_shares": {k: round(v[0] / tot, 4) for k, v in rep.items()},
           "kernel_launches_per_solve": launches, "gpu_kernel_ms_per_solve": tot,
           "roofline": {"bound": "hbm", "kernel": "ba_lm_kernel (whole two-stage solve, one launch)", "achieved": (its / reps) * bpi / (dt / reps) / 1e9,
                        "peak": peak, "unit": "GB/s", "frac": (its / reps) * bpi / (dt / reps) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                        "note": "one C3 window is 0.66 MB per LM iteration and lives in L2: a single solve is barrier/latency bound "
                                "(SURVEY.md 7 'hard parts'); the HBM roofline is meaningful for the batched and C5 legs"}}
    # ---- batched: K independent windows per launch (8 distinct windows tiled).  K = 296 fills the GPU's resident CTA slots
    #      (2 per SM x 148).  Two host threads, each with its own context, alternate: while one thread's launch runs, the other
    #      packs / unpacks its windows (ctypes releases the GIL inside the ABI call) - the same idea as the front-end's e2e chunks.
    try:
        import threading
        K, T = 296, 2
        base = [synth.make_ba_problem(100 + i, 10, 2000, 8000) for i in range(8)]
        mk = lambda: [clone(base[i % 8]) for i in range(K)]
        for _ in range(2):
            api.local_ba_batch(ctx, mk())
        breps = 4
        sets = [mk() for _ in range(breps)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bits = 0
        for st in sets:
            rs, _ = api.local_ba_batch(ctx, st)
            bits += sum(r["iters_robust"] + r["iters_refine"] for r in rs)
        torch.cuda.synchronize()
        bdt1 = time.perf_counter() - t0
        one_thread = K * breps / bdt1
        ctx.profile(True)
        api.local_ba_batch(ctx, mk())
        krep = ctx.profile_report()
        ctx.profile(False)
        kernel_ms = sum(v[0] for v in krep.values())
        ctxs = [api.Context(ctx.device) for _ in range(T)]              # one context (stream, pinned staging) per host thread
        for c in ctxs:
            for _ in range(2):
                api.local_ba_batch(c, mk())
        tsets = [[mk() for _ in range(breps)] for _ in range(T)]
        tbits = [0] * T

        def work(ti):
            for st in tsets[ti]:
                rs, _ = api.local_ba_batch(ctxs[ti], st)
                tbits[ti] += sum(r["iters_robust"] + r["iters_refine"] for r in rs)

        torch.cuda.synchronize()
        th = [threading.Thread(target=work, args=(ti,)) for ti in range(T)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        for c in ctxs:
            c.sync()
        bdt = time.perf_counter() - t0
        nsolve = K * breps * T
        ach = sum(tbits) * bpi / bdt / 1e9
        out["batched"] = {"value": nsolve / bdt, "unit": "solves/s", "windows_per_launch": K, "host_threads": T,
                          "ms_per_launch": 1e3 * bdt / (breps * T), "one_thread_value": one_thread,
                          "kernel_ms_per_launch": kernel_ms, "kernel_only_value": K / (kernel_ms * 1e-3) if kernel_ms > 0 else None,
                          "lm_iterations_per_solve": sum(tbits) / nsolve,
                          "roofline": {"bound": "hbm", "kernel": "ba_lm_kernel (K windows per launch)", "achieved": ach, "peak": peak, "unit": "GB/s",
                                       "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                                       "algorithmic_bytes": "67 N_obs + 64 N_pts per LM iteration x iterations run (SURVEY 8d)"}}
    except Exception as e:
        out["batched"] = {"error": str(e)[:200]}
    try:
        from oracle import ba_ref_c
        ts = []
        for _ in range(10):
            pb = clone()
            t = time.perf_counter()
            r = ba_ref_c.local_ba(pb)
            ts.append(time.perf_counter() - t)
        out["cpu_baseline"] = {"value": 1.0 / float(np.median(ts)), "unit": "solves/s", "cores": 1, "kind": "port",
                               "sample": "10 solves of the same C3 problem, oracle/ba_ref_c.c single thread (restatement, not Ceres; "
                                         "the reference sets num_threads = 1)", "lm_iterations": r["iters_robust"] + r["iters_refine"]}
    except Exception as e:
        out["cpu_baseline"] = {"error": str(e)[:120]}
    return out


def class_path_bench():
    """The reference-facing CLASS boundary, one frame per call (host/shim_selftest --bench): what a single live camera
    stream sees through FeatureTracker / FeatureExtractor on one GPU (every call synchronises; each image uploaded once
    thanks to the shims' device-pyramid cache).  Latency bound by construction - the batch ABI above is the throughput path."""
    from ov2slam_b200 import build, synth
    exe = build.LIB / "shim_selftest"
    if not exe.exists():
        return {"error": "shim_selftest not built"}
    n = 24
    frames = [synth.make_frame(900, W_IMG, H_IMG)]
    rng = np.random.default_rng(9)
    for k in range(1, n):                                   # a smooth synthetic sequence: small translations + noise
        sh = synth.shift_image(frames[-1], float(rng.uniform(-3, 3)), float(rng.uniform(-3, 3))) + rng.normal(0, 1.5, (H_IMG, W_IMG))
        frames.append(np.clip(np.rint(sh), 0, 255).astype(np.uint8))
    with tempfile.NamedTemporaryFile(suffix=".raw", delete=False) as f:
        f.write(np.ascontiguousarray(np.stack(frames)).tobytes())
        path = f.name
    try:
        out = subprocess.run([str(exe), "--bench", path, str(W_IMG), str(H_IMG), str(n), "20"], capture_output=True, text=True, timeout=300)
    finally:
        os.unlink(path)
    if out.returncode != 0:
        return {"error": (out.stderr or out.stdout)[-200:]}
    tok = out.stdout.split()
    d = {tok[i]: float(tok[i + 1]) for i in range(1, len(tok) - 1, 2)}
    return {"value": d.get("fps"), "unit": "frames/s", "frames": int(d.get("frames", 0)), "tracked_per_frame": d.get("tracked_per_frame"),
            "detected_per_frame": d.get("detected_per_frame"),
            "what": "FeatureTracker::fbKltTracking x2 + describeBRIEF + detectGridFAST + describeBRIEF per 640x480 frame through the C++ drop-in "
                    "classes, one stream, one frame per call"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="frame pairs per GPU per step")
    ap.add_argument("--e2e-stepped", action="store_true", help="headline e2e with a barrier after every step (default: pipelined)")
    ap.add_argument("--kernels-only", action="store_true", help="run the resident steps only and exit (for ncu captures)")
    ap.add_argument("--e2e-chunks", type=int, default=0,
                    help="chunks (host threads x contexts) of the e2e arm; 0 = 8 on one GPU, fewer per rank when several "
                         "ranks share the host cores")
    ap.add_argument("--only", default="c2", choices=["c2", "c4", "c5"], help="with --kernels-only: which leg's resident steps to run")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-ba", action="store_true", help="skip the local-BA (C3) leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 (stereo 1280x720) leg")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 (localBA 150k observations) leg")
    ap.add_argument("--c4-batch", type=int, default=144, help="stereo units per GPU per C4 step (144: every SM has a frame in the one-CTA-per-frame detector sweep)")
    ap.add_argument("--c4-unique", type=int, default=16, help="generated C4 units (the rest of the batch are flips / repeats)")
    ap.add_argument("--c4-steps", type=int, default=10)
    ap.add_argument("--c5-reps", type=int, default=5)
    ap.add_argument("--c5-small", action="store_true", help="20 KF x 3000 pts x 18000 obs instead of the C5 window (debugging)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed front-end step computed to DIR/<name>.npy "
                                                          "(float32, at most 64 MB; the inputs are the same from run to run)")
    args = ap.parse_args()
    if args.impl == "reference":
        return reference_arm(args)
    return gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
