#!/usr/bin/env python
"""bench.py -- disparity volumes/s of the STEREO_GIF hot path (CVC -> CVF -> WTA) on B200.

Contract (see the task brief): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line
on rank 0.  A "step" is one stereo frame through CostConst_GPU + CostFilter_GPU + DispSelect_GPU
producing BOTH disparity maps.  Workload at every N: BASELINE config C4, synthetic 1920x1080, D=128,
fp32 (`--workload C3|C5` select the other synthetic BASELINE configs).  N>1 (launched by torchrun, one
rank per GPU): the disparity axis is sharded D/N slices per rank; the one exchange of the path (per-pixel
packed (cost,d) minima -> final maps) is a fused reduce-scatter + all-gather over NVLink peer memory
(strong scaling: the frame is fixed, `value` = frames/s of the whole job).

  value    : frames/s with the interleaved f32 images already resident in HBM (device-timed, CUDA events)
  e2e      : same metric through the host-facing C-ABI calls: frames in pinned HOST memory, the H2D copy of
             every frame's two images and the D2H read of both u8 maps inside the timed region (the upload
             of frame k+1 overlaps the computation of frame k: psm_set_images_async)
  roofline : the fused CVF kernel's algorithmic bytes / its event-timed duration vs the measured HBM peak,
             plus the pipe that actually limits it (from the committed ncu summary)
  parity   : before the line is printed, the maps fetched by the last e2e step are compared with the CPU
             oracle on a row band (exact mode: equal; mixed mode: +-1, flips counted)
  cpu_baseline / --impl reference : the reference's pthreads CPU path on the host cores: oracle/_ref (the
             reference's own CVC/CVF/DispSel sources compiled against an OpenCV shim) when it was built,
             else the C port; a bounded slice sample per step, all cores and the reference's 8-thread cap

--dump-outputs DIR writes what the timed path computed in its last step (both disparity maps, float32 .npy); the
frame is generated from a fixed seed per workload, so two builds can be compared output for output.
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

WORKLOADS = {  # BASELINE.json configs; C4 is the one the metric is quoted on and the default at every N
    "C3": (1280, 720, 64), "C4": (1920, 1080, 128), "C5": (1920, 1080, 256),
}
METRIC = "disparity_volumes_per_s"
UNIT = "volumes/s"
MODES = ["exact", "mixed", "naive"]


def workload_name(key):
    W, H, D = WORKLOADS[key]
    return f"{key} synthetic {W}x{H} D={D} fp32, both views (lDisMap+rDisMap)"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_facts(workload, mode):
    """ncu-derived facts for THIS workload and mode from the committed summary (profiles/cvf_profile_facts.json):
    DRAM traffic per launch and the limiting pipe.  None when that combination was never profiled."""
    p = os.path.join(ROOT, "profiles", "cvf_profile_facts.json")
    try:
        return json.load(open(p)).get(f"{workload}:{mode}")
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
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
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU side (test infrastructure used as the reported baseline / the checker, never as the product path)
# ------------------------------------------------------------------------------------------------------
def cpu_backend():
    """-> (kind, pipeline(l, r, D, threads) -> dict with times_ms)"""
    from oracle import ref as R
    if R.available():
        return "reference", lambda l, r, D, threads: R.pipeline(l, r, D, threads=threads)
    from oracle import oracle as O
    return "port", lambda l, r, D, threads: O.pipeline(l, r, D, threads=threads)


def cpu_sample(run, l, r, D, threads, slices):
    """CVC+CVF+WTA of the first `slices` disparity slices of both views on `threads` host threads
    -> seconds extrapolated to the full frame (per-slice work is uniform; WTA is ~1 % of a frame)."""
    t0 = time.perf_counter()
    res = run(l, r, slices, threads)
    dt = time.perf_counter() - t0
    return dt * (D / slices), res["times_ms"]


def cpu_report(l, r, D, workload, steps, warmup):
    """The CPU arm: `steps` timed samples at all host cores (after `warmup`), plus one sample at the reference's
    own cap of 8 threads (MAX_CPU_THREADS, include/ComFunc.h:52).  Sample = min(threads, D) slices per view so
    that one batch of the reference's one-thread-per-slice scheduler is timed (DispEst.cpp:235-251)."""
    kind, run = cpu_backend()
    cores = os.cpu_count() or 1
    th_all = min(cores, D)
    s_all = min(D, max(th_all, 16))
    for _ in range(warmup):
        cpu_sample(run, l, r, D, th_all, s_all)
    ts = [cpu_sample(run, l, r, D, th_all, s_all)[0] for _ in range(max(1, steps))]
    sec = float(np.mean(ts))
    th8 = min(8, cores)
    sec8, _ = cpu_sample(run, l, r, D, th8, th8)
    what = ("reference's own src/{CVC,CVF,DispSel}.cpp compiled against oracle/shim (oracle/_ref)" if kind == "reference"
            else "C port of the reference path (oracle/libstereo_oracle.so; oracle/_ref not built)")
    return {
        "value": 1.0 / sec, "unit": UNIT, "cores": th_all, "kind": kind,
        "sample": f"{s_all} of {D} disparity slices of both views of {workload} on {th_all} threads, scaled x{D / s_all:g}; {what}",
        "host_cores": cores,
        "capped_8_threads": {"value": 1.0 / sec8, "unit": UNIT, "cores": th8,
                             "sample": f"{th8} of {D} slices on {th8} threads (the reference's MAX_CPU_THREADS cap), scaled x{D / th8:g}"},
    }, sec


def run_reference(args, rank):
    """--impl reference: the reference's CPU path on the host cores, rank 0 only."""
    if rank != 0:
        return
    from primestereomatch_b200 import synth
    W, H, D = WORKLOADS[args.workload]
    l, r, _ = synth.stereo_pair_f32(W, H, D)
    cb, sec = cpu_report(l, r, D, workload_name(args.workload), args.steps, args.warmup)
    val = 1.0 / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload)},
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def oracle_band_maps(l, r, D, y0, y1):
    """Both disparity maps of rows [y0, y1) from the CPU oracle run on a row band with a 16-row margin (8 rows
    of guide means + 8 of the two box stages reach into the neighbourhood; image borders reflect as in the frame)."""
    from oracle import oracle as O
    H = l.shape[0]
    c0, c1 = max(0, y0 - 16), min(H, y1 + 16)
    res = O.pipeline(np.ascontiguousarray(l[c0:c1]), np.ascontiguousarray(r[c0:c1]), D, threads=min(os.cpu_count() or 1, D))
    return res["lDis"][y0 - c0:y1 - c0], res["rDis"][y0 - c0:y1 - c0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cvf-mode", type=int, default=0, help="0 exact (default, the headline), 1 mixed (tolerance mode)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS),
                    help="C4 (default) is the benchmark; C3 / C5 are the other synthetic BASELINE configs")
    ap.add_argument("--seg-rows", type=int, default=0)
    ap.add_argument("--extra-smem", type=int, default=0)
    ap.add_argument("--cta-threads", type=int, default=0)
    ap.add_argument("--remap", type=int, default=0)
    ap.add_argument("--emulate-shards", type=int, default=1,
                    help="tuning: one GPU runs the per-rank share (D/N slices, no exchange) of an N-GPU run; not a benchmark line")
    ap.add_argument("--cvc-chunk", type=int, default=0, help="slices per CTA of the CVC kernel (tuning A/B, option 108)")
    ap.add_argument("--guide-rows", type=int, default=0, help="rows per warp of the guide precompute (tuning A/B, option 107)")
    ap.add_argument("--cvc-variant", type=int, default=0, help="CVC kernel build (tuning A/B, option 106)")
    ap.add_argument("--no-pack", type=int, default=0, help="1: one warp per slice for the last W %% 112 columns (tuning A/B)")
    ap.add_argument("--upload", default="banded", choices=["banded", "replicated"],
                    help="N>1, e2e: banded = every rank uploads H/N rows of both images and the bands are "
                         "all-gathered over NVLink; replicated = every rank uploads both full images over PCIe")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "p2p-barrier", "nccl"],
                    help="N>1: p2p = fused WTA + exchange over NVLink peer memory, ordered by device-side flags; "
                         "p2p-barrier = same kernels separated by NCCL barriers; nccl = local WTA then ncclAllGather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the disparity maps of the last timed step as DIR/lDisMap.npy and "
                         "DIR/rDisMap.npy (float32, H x W) on rank 0, to compare two builds on the same seeded frame")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.emulate_shards > 1):
        ap.error("--dump-outputs needs the product path (--impl ours) without --emulate-shards")
    W, H, D = WORKLOADS[args.workload]
    WORKLOAD = workload_name(args.workload)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return 0

    import torch
    import torch.distributed as dist
    from primestereomatch_b200 import DispEst, capi, synth
    from primestereomatch_b200.sharding import BandedUpload, P2PExchange, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus or world == 1, (world, args.gpus)
    warm = max(3, args.warmup)

    L = capi.lib()
    l8, r8, _ = synth.stereo_pair_u8(W, H, D)
    l, r = synth.to_f32(l8), synth.to_f32(r8)
    lp8 = torch.from_numpy(l8).pin_memory()
    rp8 = torch.from_numpy(r8).pin_memory()
    lp = torch.from_numpy(l).pin_memory()
    rp = torch.from_numpy(r).pin_memory()
    ld_dev, rd_dev = lp.cuda(), rp.cuda()
    torch.cuda.synchronize()

    d_begin, d_count = shard_range(D, world, rank)
    if args.emulate_shards > 1:
        assert world == 1
        d_begin, d_count = shard_range(D, args.emulate_shards, 0)
        args.no_parity = True
    de = DispEst(l, r, D, 8, True, device=local_rank, d_begin=d_begin, d_count=d_count)
    de.set_option(capi.PSM_OPT_CVF_MODE, args.cvf_mode)
    de.set_option(capi.PSM_OPT_VARIANT, args.variant)
    de.set_option(101, args.seg_rows)
    de.set_option(102, args.extra_smem)
    de.set_option(103, args.cta_threads)
    de.set_option(104, args.remap)
    de.set_option(105, args.no_pack)
    de.set_option(106, args.cvc_variant)
    de.set_option(107, args.guide_rows)
    de.set_option(108, args.cvc_chunk)
    stream = torch.cuda.Stream()  # a real (non-default) stream shared by the context and torch's collectives
    torch.cuda.set_stream(stream)
    capi.check(L.psm_set_stream(de.handle, C.c_void_p(stream.cuda_stream)), de.handle)

    npix = W * H
    lmap = torch.empty((H, W), dtype=torch.uint8).pin_memory()
    rmap = torch.empty((H, W), dtype=torch.uint8).pin_memory()
    p2p = None
    if world > 1 and args.exchange == "nccl":
        keys = torch.empty((2, npix), dtype=torch.int64, device="cuda")
        gathered = torch.empty((2, world, npix), dtype=torch.int64, device="cuda")
    elif world > 1:
        p2p = P2PExchange(de, world, rank, device_sync=(args.exchange == "p2p"))
    emu_keys = torch.empty((2, npix), dtype=torch.int64, device="cuda") if args.emulate_shards > 1 else None
    step_bytes = W * 3 * 4
    banded = BandedUpload(de, world, rank) if (world > 1 and args.upload == "banded") else None

    def finish(e2e):
        """stages after the images are set: CVC, CVF, WTA (+ exchange), maps to host when e2e"""
        capi.check(L.psm_cost_const(de.handle), de.handle)
        capi.check(L.psm_cost_filter(de.handle), de.handle)
        if args.emulate_shards > 1:   # tuning: the rank's local WTA, no exchange
            capi.check(L.psm_disp_select_keys(de.handle, emu_keys[0].data_ptr(), emu_keys[1].data_ptr()), de.handle)
        elif world == 1:
            if e2e:  # D2H enqueued, not synchronised: the host maps are read after the timed region's final sync
                capi.check(L.psm_disp_select_async(de.handle, lmap.data_ptr(), W, rmap.data_ptr(), W), de.handle)
            else:
                capi.check(L.psm_disp_select_device(de.handle), de.handle)
        elif p2p is not None:
            p2p.frame(lmap.data_ptr() if e2e else None, rmap.data_ptr() if e2e else None)
        else:
            capi.check(L.psm_disp_select_keys(de.handle, keys[0].data_ptr(), keys[1].data_ptr()), de.handle)
            dist.all_gather_into_tensor(gathered[0].view(-1), keys[0])
            dist.all_gather_into_tensor(gathered[1].view(-1), keys[1])
            out_l = lmap.data_ptr() if e2e else None
            out_r = rmap.data_ptr() if e2e else None
            capi.check(L.psm_disp_reduce_keys(de.handle, gathered[0].data_ptr(), gathered[1].data_ptr(), world,
                                              out_l, W, out_r, W), de.handle)

    def upload_async(e2e):
        if e2e == "u8":
            capi.check(L.psm_set_images_u8_async(de.handle, lp8.data_ptr(), W * 3, rp8.data_ptr(), W * 3), de.handle)
        else:
            capi.check(L.psm_set_images_async(de.handle, lp.data_ptr(), step_bytes, rp.data_ptr(), step_bytes), de.handle)

    def run_steps(e2e, n):
        """n frames.  Device-resident inputs (e2e False): ingest from HBM.  Host frames: at N=1 (and N>1 replicated)
        a two-deep pipeline -- the H2D of frame k+1 runs on the copy stream while frame k computes; banded N>1:
        the same pipeline with band upload + NVLink all-gather on a side stream."""
        if not e2e:
            for _ in range(n):
                capi.check(L.psm_set_images_device(de.handle, ld_dev.data_ptr(), step_bytes, rd_dev.data_ptr(), step_bytes), de.handle)
                finish(False)
        elif banded is not None and e2e != "u8":
            banded.upload_async(lp, rp)        # frame 0: band H2D + NVLink all-gather on the side stream
            for k in range(n):
                banded.commit()
                if k + 1 < n:
                    banded.upload_async(lp, rp)
                finish(True)
        else:
            upload_async(e2e)                  # frame 0
            for k in range(n):
                capi.check(L.psm_set_images_commit(de.handle), de.handle)
                if k + 1 < n:
                    upload_async(e2e)          # frame k+1 uploads while frame k computes
                finish(True)

    def timed(e2e, steps):
        """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launching
        stream, max over ranks.  No host synchronisation inside the region."""
        run_steps(e2e, warm)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_steps(e2e, steps)
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def kernel_times(steps):
        """Duration of the fused CVF kernel alone (cudaEvent pair around that launch, on the launching
        stream) for `steps` further steps of the same workload; reading an event pair needs a host
        sync per step, which is why this is a separate loop from the throughput measurement."""
        out = []
        for _ in range(steps):
            run_steps(False, 1)
            out.append(de.stage_ms(4))
        return out

    def dump_maps(out_dir):
        """Both u8 disparity maps of the last step, read where that step left them (the context's device maps; with
        the fused p2p exchange, the complete maps in the exchange block), saved as float32 .npy."""
        if p2p is not None:
            p2p.fetch(lmap.data_ptr(), rmap.data_ptr())
            de.sync()
            maps = [lmap.numpy().copy(), rmap.numpy().copy()]
        else:
            maps = []
            for what in (2, 3):
                ptr, pitch = C.c_void_p(), C.c_size_t()
                capi.check(L.psm_device_ptr(de.handle, what, C.byref(ptr), C.byref(pitch)), de.handle)
                view = type("DeviceMap", (), {"__cuda_array_interface__": {
                    "shape": (H, W), "typestr": "|u1", "data": (ptr.value, False), "strides": (pitch.value, 1),
                    "version": 2}})()
                maps.append(torch.as_tensor(view, device="cuda").cpu().numpy())
        os.makedirs(out_dir, exist_ok=True)
        for name, m in zip(("lDisMap", "rDisMap"), maps):
            np.save(os.path.join(out_dir, f"{name}.npy"), m.astype(np.float32))

    launches0 = de.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms = timed(False, args.steps)
    launches_per_step = (de.launch_count() - launches0) // (warm + args.steps)
    if args.dump_outputs and rank == 0:
        dump_maps(args.dump_outputs)
    kms = kernel_times(args.steps)
    clocks = sampler.stop() if rank == 0 else None
    stage = {n: de.stage_ms(i) for i, n in enumerate(["ingest", "cvc", "cvf", "wta", "cvf_kernel"])}
    if args.emulate_shards > 1:
        print(json.dumps({"NOTE": "tuning run (one GPU runs the share of one rank of an N-GPU run, no exchange); not a benchmark line",
                          "workload": WORKLOAD, "emulated_share_of": args.emulate_shards, "slices": d_count,
                          "cvf_mode": MODES[args.cvf_mode], "ms_per_step": total_ms / args.steps,
                          "cvf_kernel_ms": float(np.mean(kms)), "stage_ms_last_step": stage}), flush=True)
        de.close()
        return 0
    e2e_ms = timed(True, args.steps)
    e2e_u8_ms = timed("u8", args.steps)

    # ---- parity: the maps the last timed e2e step left in host memory vs the CPU oracle on a row band ----
    parity = None
    if not args.no_parity:
        run_steps(True, 1)
        torch.cuda.synchronize()
        if rank == 0:
            y0, y1 = H // 2 - 24, H // 2 + 24
            wl, wr = oracle_band_maps(l, r, D, y0, y1)
            gl, gr = lmap.numpy()[y0:y1], rmap.numpy()[y0:y1]
            dl = np.abs(gl.astype(np.int16) - wl.astype(np.int16))
            dr = np.abs(gr.astype(np.int16) - wr.astype(np.int16))
            worst = int(max(dl.max(), dr.max()))
            flips = int((dl > 0).sum() + (dr > 0).sum())
            ok = worst == 0 if args.cvf_mode == 0 else worst <= 1
            parity = {"checked": True, "ok": bool(ok), "rows": [y0, y1], "max_abs_disparity_diff": worst,
                      "pixels_differing": flips, "against": "CPU oracle (oracle/libstereo_oracle.so) on the same frame",
                      "rule": "equal" if args.cvf_mode == 0 else "+-1 disparity level"}
            if not ok:
                raise SystemExit(f"bench.py: PARITY FAILURE against the oracle: {parity}")

    # ---- the tolerance mode north_star allows for fp32 (a, b exact; fp32 second box stage), same run, same frame ----
    mixed = None
    if world == 1 and args.cvf_mode == 0:
        run_steps(True, 1)
        torch.cuda.synchronize()
        exact_l, exact_r = lmap.numpy().copy(), rmap.numpy().copy()
        de.set_option(capi.PSM_OPT_CVF_MODE, 1)
        m_ms = timed(False, args.steps)
        m_kms = float(np.mean(kernel_times(args.steps)))
        run_steps(True, 1)
        torch.cuda.synchronize()
        dl = np.abs(lmap.numpy().astype(np.int16) - exact_l.astype(np.int16))
        dr = np.abs(rmap.numpy().astype(np.int16) - exact_r.astype(np.int16))
        mixed = {"cvf_mode": MODES[1], "value": 1e3 / (m_ms / args.steps), "unit": UNIT, "ms_per_step": m_ms / args.steps,
                 "kernel_ms": m_kms, "maps_vs_exact": {"max_abs_disparity_diff": int(max(dl.max(), dr.max())),
                                                       "pixels_differing": int((dl > 0).sum() + (dr > 0).sum()),
                                                       "pixels": int(2 * W * H)}}
        if mixed["maps_vs_exact"]["max_abs_disparity_diff"] > 1:
            raise SystemExit(f"bench.py: PSM_CVF_MIXED left its +-1 disparity tolerance: {mixed}")
        de.set_option(capi.PSM_OPT_CVF_MODE, 0)

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = 1e3 / ms_per_step
        e2e_value = 1e3 / (e2e_ms / args.steps)
        peak, peak_src = measured_peaks()
        V = W * H * d_count
        algo_bytes = 2 * (8 * V + 48 * W * H)  # one launch filters both views: read p + write q + 12 guide floats/px
        kern_ms = float(np.mean(kms))
        achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
        mode = MODES[args.cvf_mode]
        facts = profile_facts(args.workload, mode) if world == 1 else None
        h2d = banded.h2d_bytes() if banded is not None else 2 * W * H * 3 * 4
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "parallelism": (f"disparity-sharded x{world}, exchange={args.exchange}") if world > 1 else "single GPU",
                       "cvf_mode": mode, "variant": args.variant,
                       **({"emulated_share_of": args.emulate_shards, "NOTE": "tuning run, not a benchmark line"} if args.emulate_shards > 1 else {}),
                       "l2": f"inputs larger than L2: each step streams {4 * V * 4 / 1e9:.2f} GB of volumes (raw+filtered, 2 views) per GPU"
                             + ("" if 4 * V * 4 > 252e6 else "; NOTE: smaller than 2 x L2, L2 reuse between steps is possible"),
                       "stage_ms_last_step": stage},
            "roofline": {"bound": "hbm", "kernel": "cvf_stream_kernel (fused guided filter, both views per launch)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (facts or {}).get("dram_bytes_per_launch"),
                         "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": kern_ms, "peak_source": peak_src,
                         "limiter": (facts or {}).get("limiter",
                                                      "not profiled for this workload/mode; see profiles/ for C4")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
                    "upload": ("banded, two-deep pipeline: each rank uploads H/N rows, NCCL all-gather over NVLink, on a side stream" if banded is not None
                               else "two-deep pipeline: frame k+1 uploads (copy stream) while frame k computes"),
                    "d2h_bytes_per_step": 2 * W * H * world, "ms_per_step": e2e_ms / args.steps},
            "e2e_u8": {"value": 1e3 / (e2e_u8_ms / args.steps), "unit": UNIT, "h2d_bytes_per_step": 2 * W * H * 3 * world,
                       "d2h_bytes_per_step": 2 * W * H * world, "ms_per_step": e2e_u8_ms / args.steps,
                       "note": "same as e2e but the host frames are 8-bit (psm_set_images_u8_async)"},
            "gpu_launches": int(launches_per_step * args.steps),
            "parity_checked": bool(parity and parity["ok"]),
            "parity": parity,
            "clocks": clocks,
        }
        if facts and "executed_warp_instructions" in facts:
            # what actually binds: the instruction stream at 12 warps per SM.  Live: warp instructions of the profiled launch
            # (committed ncu summary of this workload and mode) / the kernel time measured in THIS run, against 4 warp
            # instructions per clock per SM at the SM clock sampled in this run.
            sm_mhz = float((clocks or {}).get("sm_mhz") or 1965.0)
            peak_ips = 148 * 4 * sm_mhz * 1e6
            ips = facts["executed_warp_instructions"] / (kern_ms * 1e-3)
            line["roofline"]["issue"] = {"achieved": ips / 1e12, "peak": peak_ips / 1e12, "unit": "T warp-instructions/s",
                                         "frac": ips / peak_ips, "issue_active_pct_in_profile": facts.get("issue_active_pct"),
                                         "warps_per_sm": facts.get("warps_per_sm"),
                                         "note": "instruction count from the committed ncu capture of this workload/mode; time and clock from this run"}
        if mixed is not None:
            mixed["roofline_frac"] = algo_bytes / (mixed["kernel_ms"] * 1e-3) / 1e9 / peak
            line["tolerance_mode"] = mixed
        if world == 1 and not args.no_cpu_baseline:
            cb, _ = cpu_report(l, r, D, WORKLOAD, steps=1, warmup=1)
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    de.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
