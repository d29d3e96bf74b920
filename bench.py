#!/usr/bin/env python
"""bench.py -- headline benchmark of the DAGR hot path on B200 (contract: see the task statement).

  python bench.py --gpus N --steps K --warmup W            # ours (sm_100a kernels)
  python bench.py --impl reference --steps K --warmup W    # reference-equivalent CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Headline workload (BASELINE.json configs[1]): dagr-s, events only, synthetic DSEC-shaped 640x480 streams,
50 ms window, 300k events/sample, batch 8 per GPU.  A "step" is one synchronous forward
(graph build -> SplineConv layers -> voxel pooling -> head -> decode -> NMS [-> NCCL detection
all-gather when N > 1]).  `value` = events of all ranks / step time with inputs resident in HBM;
`e2e` = the same through the public API (format_data + DAGR.forward) from pinned HOST buffers with the
H2D copy and the detection read-back inside the timed region.

The same JSON line also carries the rest of BASELINE.json's story (all measured in the default run):
  clustered              the headline loop on the clustered stream (moving edge segments + noise, SURVEY 8d)
  sustained              >= 2 s of back-to-back steps with clock samples
  interframe_latency_ms  config 3: dagr-s + ResNet-50 image fusion, run_test_interframe windows, B = 8 and B = 1
  streaming              config 5: dagr-l, one 1 Mevents/s stream in 1 ms chunks, 50 ms live window, >= 2 s of stream
  extra.config4          (N > 1 only) dagr-m, batch 8 per GPU
"""
import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch

W, H, T = 640, 480, 1_000_000
METRIC, UNIT = "Mevents/sec", "Mevents/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--size", default="s")
    p.add_argument("--batch", type=int, default=8, help="samples per GPU")
    p.add_argument("--events", type=int, default=300_000, help="events per sample")
    p.add_argument("--kind", default="uniform", choices=["uniform", "clustered"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-overlap", action="store_true", help="serial steps (no side-stream overlap of consecutive forwards)")
    p.add_argument("--cpu-seconds", type=float, default=20.0, help="target CPU work for the baseline sample")
    p.add_argument("--sustained-seconds", type=float, default=2.0)
    p.add_argument("--headline-only", action="store_true", help="skip clustered / sustained / config 3 / config 5 / config 4")
    p.add_argument("--stream-seconds", type=float, default=2.0, help="length of the config-5 stream")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the headline loop returned (decoded "
                                                         "outputs, detections) as DIR/<name>.npy, to compare two builds")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be >= 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs applies to the GPU arm (--impl ours)")
    return a


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """samples SM clocks / throttle reasons during the timed region (NVML, 20 ms period)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            while not self.stop_flag:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = get_reasons(h)
                self.rows.append((mhz, [k for k, bit in names.items() if r & bit]))
                time.sleep(0.02)
        except Exception as e:                                   # pragma: no cover
            self.rows.append((None, [f"nvml unavailable: {e}"]))

    def mark(self):
        return len(self.rows)

    def summary(self, lo=0, hi=None):
        rows = self.rows[lo:hi]
        sm = sorted(r[0] for r in rows if r[0] is not None)
        reasons = sorted({x for r in rows for x in r[1]})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=self.max_mhz, reasons=reasons, samples=len(rows))


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        j = json.loads(f.read_text())
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
def crop_sample(raw, frac_events):
    """bounded CPU sample: events of sample 0 inside a centred crop holding ~frac of them, so that the
    local event density (hence the neighbour degree, hence the per-event cost) is that of the full workload."""
    import math
    m = raw.batch == 0
    xy, t, p = raw.pos[m], raw.t[m], raw.x[m]
    s = math.sqrt(max(min(frac_events, 1.0), 1e-4))
    w, h = max(16, int(W * s)), max(16, int(H * s))
    x0, y0 = (W - w) // 2, (H - h) // 2
    k = (xy[:, 0] >= x0) & (xy[:, 0] < x0 + w) & (xy[:, 1] >= y0) & (xy[:, 1] < y0 + h)
    return xy[k], t[k], p[k], (w, h)


_REF_CACHE = {}


def _ref_model(model_sd, margs):
    """one RefModel per process: its per-conv LUTs are built once (the reference's cache_luts is a
    one-off too, run_test.py:59) and are not part of the timed forward."""
    from oracle.ref_model import RefModel
    if "m" not in _REF_CACHE:
        _REF_CACHE["m"] = RefModel(model_sd, margs, H, W)
    return _REF_CACHE["m"]


def cpu_reference_run(model_sd, margs, raw, n_target, steps, warmup, threads):
    """times the oracle restatement of the reference's forward on host cores."""
    from oracle import ref_ops as R
    torch.set_num_threads(threads)
    nfull = int((raw.batch == 0).sum())
    xy, t, p, crop = crop_sample(raw, n_target / nfull)
    pos = R.format_pos(xy, t, W, H, T)
    x = p.float()
    batch = torch.zeros(len(x), dtype=torch.long)
    ref = _ref_model(model_sd, margs)
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ref.forward(x, pos, batch, 1)
        ts.append(time.perf_counter() - t0)
    ts = ts[warmup:]
    sec = sum(ts) / len(ts)
    return dict(events=len(x), sec_per_step=sec, mev_s=len(x) / sec / 1e6, threads=threads, crop=crop,
                sample=f"B = 1: sample 0 of the workload cropped to {crop[0]}x{crop[1]} px at full event density "
                       f"({len(x)} events), full 640x480 dagr-{margs_size(margs)} forward incl. NMS; LUTs pre-built")


def cpu_calibrate(model_sd, margs, raw):
    """builds the LUT caches (untimed) and picks the torch thread count that is fastest on a small sample."""
    cpu_reference_run(model_sd, margs, raw, 3000, 1, 0, min(os.cpu_count() or 1, 16))       # LUT build, untimed
    best = None
    for th in sorted({min(os.cpu_count() or 1, c) for c in (8, 32, os.cpu_count() or 1)}):
        r = cpu_reference_run(model_sd, margs, raw, 6000, 1, 1, th)
        if best is None or r["sec_per_step"] < best["sec_per_step"]:
            best = r
    return best


def margs_size(a):
    return {0.25: "n", 0.5: "s", 0.75: "m", 1.0: "l"}.get(float(a.net_stem_width), "?")


def _pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(q * len(xs)))]


def host_outputs(dec, det, ndet):
    """one step's results on the host: decoded [B, anchors, 5 + classes] (forward_decoded), detections [B, anchors, 6]
    (x1, y1, x2, y2, score, label; the NMS kernel leaves the rows past num_detections unwritten, they are stored as 0) and
    num_detections [B]."""
    det, ndet = det.float().cpu(), ndet.cpu()
    for b in range(len(ndet)):
        det[b, int(ndet[b]):] = 0
    return dict(decoded=dec.float().cpu().numpy(), detections=det.numpy(), num_detections=ndet.double().numpy())


# ------------------------------------------------------------------------------------------------
def measure_interframe(a, dev):
    """config 3 (BASELINE.json configs[2], scripts/run_test_interframe.py:83-86): dagr-s + ResNet-50 image fusion, the
    synchronous forward on windows of growing length num_us = linspace(0, 50 ms, 10), for B = batch and B = 1."""
    import numpy as np
    from dagr_b200.data import EventBatch, format_data, synth_batch
    from dagr_b200.model.dagr import DAGR
    from dagr_b200.utils.args import default_args
    from tests.helpers import randomize_bn
    out = {}
    for B in sorted({a.batch, 1}, reverse=True):
        torch.manual_seed(0)
        iargs = default_args(a.size, batch_size=B, use_image=True, img_net="resnet50")
        m3 = randomize_bn(DAGR(iargs, height=H, width=W).eval()).to(dev)
        raw = synth_batch(B, a.events, W, H, seed=4242, kind=a.kind, with_image=True)
        d = format_data(raw.clone().to(dev))
        t_us = (d.pos[:, 2].double() * T).round()
        steps = []
        for n_us in np.linspace(0, 50000, 10):
            msk = t_us < (T - 50000 + n_us)
            sub = EventBatch(x=d.x[msk], pos=d.pos[msk], batch=d.batch[msk], width=d.width, height=d.height, time_window=d.time_window,
                             image=d.image, num_graphs=B, dims=(W, H, T))
            for _ in range(2):
                m3(sub.clone())
            torch.cuda.synchronize()
            reps = 3
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                m3(sub.clone())
            e1.record(); torch.cuda.synchronize()
            steps.append(dict(num_us=int(n_us), events=int(msk.sum()), ms=round(e0.elapsed_time(e1) / reps, 4)))
        ms = [s["ms"] for s in steps]
        out[f"batch{B}"] = dict(steps=steps, p50_ms=_pct(ms, 0.5), max_ms=max(ms), empty_window_ms=ms[0], full_window_ms=ms[-1])
        del m3
        torch.cuda.empty_cache()
    out["config"] = (f"dagr-{a.size} + resnet50 image fusion, {W}x{H}, {a.events} events/sample ({a.kind}) in the full window; each entry is one "
                     "synchronous DAGR.forward (image trunk + CNN head via cuDNN/TF32, graph path, NMS, detection counts read back), "
                     "CUDA-event timed, mean of 3 after 2 warm-up calls")
    return out


def measure_streaming(a, dev):
    """config 5 (BASELINE.json configs[4]): dagr-l, one stream per GPU at ~1 Mevents/s fed as 1 ms chunks, 50 ms live window."""
    from dagr_b200.streaming import stream_benchmark
    return stream_benchmark(dev, size="l", width=W, height=H, rate_ev_s=1_000_000, chunk_us=1000, window_us=50_000,
                            seconds=a.stream_seconds, kind=a.kind)


# ------------------------------------------------------------------------------------------------
def main():
    a = parse()
    from dagr_b200.data import format_data, synth_batch
    from dagr_b200.utils.args import default_args
    from tests.helpers import randomize_bn

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    margs = default_args(a.size, batch_size=a.batch)
    config = dict(workload=f"dagr-{a.size} DSEC synthetic {W}x{H}, 50 ms window, {a.events} events/sample ({a.kind}), "
                           f"batch {a.batch} per GPU, events only", global_batch=a.batch * world,
                  events_per_step=a.batch * a.events * world, parallelism=f"dp{world} (batch shards, NCCL all_gather of detections)",
                  overlap=("consecutive steps overlap: coarse stack + NMS of step i on a side stream while the event-level kernels "
                           "of step i+1 run (serial_ms_per_step is the same loop without overlap)") if not a.no_overlap else "none",
                  l2="inputs rotate over 3 distinct batches; per-step working set (ELL adjacency + activations ~0.6 GB) exceeds the 126 MB L2")

    # ---------------------------------------------------------------- reference arm (CPU) --------
    if a.impl == "reference":
        if rank != 0:
            return
        config["overlap"] = "n/a (CPU arm)"
        from dagr_b200.model.dagr import DAGR
        torch.manual_seed(0)
        model = randomize_bn(DAGR(margs, height=H, width=W).eval())
        raw = synth_batch(1, a.events, W, H, seed=42 + 1000 * 2, kind=a.kind)
        # size the per-step sample so that (steps + warmup) steps take ~2 minutes
        cal = cpu_calibrate(model.state_dict(), margs, raw)
        threads = cal["threads"]
        budget = 120.0 / max(1, a.steps + a.warmup)
        n_target = int(min(a.events, max(2000, cal["events"] * budget / max(cal["sec_per_step"], 1e-3) * 0.8)))
        r = cpu_reference_run(model.state_dict(), margs, raw, n_target, a.steps, a.warmup, threads)
        # the arm's real shape: ONE host process, one sample (B = 1), a full-density crop sized to the time budget; the value is
        # a per-event rate, so it is comparable with the GPU arm's per-event rate at N = 1 (at N > 1 it is still one host process)
        config["reference_sample"] = dict(batch=1, crop_px=list(r["crop"]), events_per_step=r["events"], processes=1, threads=threads,
                                          note="bounded sample of the workload above (same model, density and code path); "
                                               "Mevents/s is a per-event rate")
        line = dict(metric=METRIC, value=r["mev_s"], unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup,
                    ms_per_step=r["sec_per_step"] * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic", config=config, impl="reference",
                    cpu_baseline=dict(value=r["mev_s"], unit=UNIT, cores=threads, kind="port", sample=r["sample"]),
                    e2e=dict(value=r["mev_s"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm (GPU) --------------
    import torch.distributed as dist
    from dagr_b200.model.dagr import DAGR
    from dagr_b200 import parallel

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout at communicator creation: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return float(ms)
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        return float(tms.item())

    def make_workload(size, kind, seed0):
        """model + three resident batches + the step closure of one workload."""
        torch.manual_seed(0)
        wargs = default_args(size, batch_size=a.batch)
        mdl = randomize_bn(DAGR(wargs, height=H, width=W).eval()).to(dev)
        raws_ = [synth_batch(a.batch, a.events, W, H, seed=seed0 + 100 * rank + 10 * i, kind=kind) for i in range(3)]
        dev_in_ = [format_data(r.clone().to(dev)) for r in raws_]      # formatted, resident in HBM
        nev = sum(int(r.pos.shape[0]) for r in raws_) / len(raws_)

        def step_(i):
            d = dev_in_[i % len(dev_in_)]
            dec = mdl.forward_decoded(d)
            det, ndet = mdl.engine.postprocess(dec, mdl.conf_threshold, mdl.nms_threshold, W, H)
            if world > 1:
                with mdl.engine.result_stream():
                    det, ndet = parallel.all_gather_detections(det, ndet)
                mdl.engine.fence()
            return dec, det, ndet
        return mdl, raws_, dev_in_, nev, step_

    def timed(eng_, step_, nsteps, warm):
        """W warm-up steps, then exactly `nsteps` steps between barriers; CUDA events; max over ranks.
        -> (ms per step, launches, what the last step returned)"""
        for i in range(warm):
            step_(i)
        barrier()
        l0 = eng_.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(nsteps):
            out = step_(i)
        eng_.join()                                              # the last steps' side-stream work is inside the timed region
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / nsteps), eng_.launches - l0, out

    model, raws, dev_in, n_events, step = make_workload(a.size, a.kind, 42 + 1000 * 2)
    eng = model.engine
    pinned = [r.clone().pin_memory() for r in raws]                    # raw dataset dtypes in pinned host memory

    # throughput mode: the coarse stack + NMS (+ the all-gather) of step i run on the engine's side stream while the
    # event-level kernels of step i+1 already execute (Engine.overlap, double-buffered hand-off); every step still does
    # all of its work and leaves its detections in device memory
    eng.overlap = not a.no_overlap
    sampler = ClockSampler(local)
    sampler.start()
    warm = max(a.warmup, 3)
    for i in range(warm):
        step(i)
    barrier()
    c0 = sampler.mark()
    ms, launches, last = timed(eng, step, a.steps, 0)
    c1 = sampler.mark()
    value = n_events * world / (ms * 1e-3) / 1e6
    dumped = host_outputs(*last) if a.dump_outputs and rank == 0 else None   # copied now: later runs reuse the buffers

    # ---- sustained: >= 2 s of back-to-back steps (same loop, same inputs) with clock samples ----------
    sustained = None
    if not a.headline_only:
        n_sus = max(a.steps, int(a.sustained_seconds / (ms * 1e-3)) + 1)
        s0 = sampler.mark()
        sms, _, _ = timed(eng, step, n_sus, 0)
        s1 = sampler.mark()
        sustained = dict(value=n_events * world / (sms * 1e-3) / 1e6, unit=UNIT, steps=n_sus, ms_per_step=sms, seconds=sms * n_sus * 1e-3,
                         clocks=sampler.summary(s0, s1))

    # ---- latency of ONE forward (serial: no overlap between consecutive steps) --------------------
    eng.overlap = False
    serial_ms, _, _ = timed(eng, step, a.steps, 3)

    # ---- e2e through the public API from pinned host memory --------------------------------------
    from dagr_b200.pipeline import PipelinedDetector, Prefetcher
    pf = Prefetcher(pinned, dev, transform=format_data)       # H2D (+ format_data) of step i+1 overlaps step i
    eng.overlap = False
    pd = PipelinedDetector(model)                              # public throughput API: submit() / Handle.result()

    def e2e_run(nsteps):
        # every step: H2D of its inputs (Prefetcher, pinned memory), the full forward, D2H of its detections;
        # step i+1 is enqueued before the host blocks on the result of step i
        h_prev, ndet_total = None, 0
        for i in range(nsteps):
            h = pd.submit(pf.next())
            if h_prev is not None:
                ndet_total += sum(int(x["boxes"].shape[0]) for x in h_prev.result())
            h_prev = h
        ndet_total += sum(int(x["boxes"].shape[0]) for x in h_prev.result())
        return ndet_total

    def e2e_sync_step():
        out = model(pf.next())[0]                              # drop-in synchronous call: detections on the device
        return [x["boxes"].cpu() for x in out]

    e2e_run(3)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_run(a.steps)
    f1.record()
    barrier()
    ems = max_over_ranks(f0.elapsed_time(f1) / a.steps)
    for i in range(2):
        e2e_sync_step()
    barrier()
    f2, f3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f2.record()
    for i in range(a.steps):
        e2e_sync_step()
    f3.record()
    barrier()
    e2e_sync_ms = f2.elapsed_time(f3) / a.steps
    r0 = raws[0]
    h2d = sum(t.numel() * t.element_size() for t in (r0.x, r0.pos, r0.t, r0.batch, r0.width, r0.height, r0.time_window))
    A = 175
    d2h = a.batch * 4 + a.batch * A * 6 * 4
    e2e = dict(value=n_events * world / (ems * 1e-3) / 1e6, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
               ms_per_step=ems, api="PipelinedDetector.submit/result", sync_api_ms_per_step=e2e_sync_ms)

    # ---- per-kernel timing pass (CUDA events around each C-ABI call, outside the headline timing) --
    def per_op(mdl, step_, n=10):
        mdl.engine.prof = {}
        for i in range(n):
            step_(i)
        torch.cuda.synchronize()
        prof_ = mdl.engine.prof_summary()
        mdl.engine.prof = None
        L = mdl.engine.last
        N_ = L["N"]
        deg = L["ws"]["nbr"][15 * N_:16 * N_].long()
        return prof_, N_, int(deg.sum().item()) + N_                # E incl. one self loop per event (SURVEY 8: E)

    prof, N, E = per_op(model, step, min(a.steps, 10))
    peak, peak_src = peaks()
    tot_ms = sum(v["ms"] for v in prof.values())
    clocks = sampler.summary(c0, c1)
    clk_ghz = (clocks.get("sm_mhz") or 1965) / 1e3
    fp32_peak = 148 * 4 * 32 * 2 * 2 / 2 * clk_ghz / 1e3              # TFLOP/s: FFMA2 = 2 lanes x 2 flop, one warp instruction per 2 cycles per SMSP
    try:                                                        # per-launch DRAM bytes from the committed ncu capture of this command
        ncu_traffic = json.load(open(ROOT / "profiles" / "ncu_traffic.json"))
    except Exception:
        ncu_traffic = {}

    # algorithmic bytes per launch, SURVEY 8(d):
    #   l1_build  = graph_build (16 N in + 16 E out, int64 edge pairs in the reference contract) + conv_block1.conv_block1
    #               (Cin 3 -> 16: 12 N + 64 N + 8 E + 4 N)                                   = 96 N + 24 E
    #   conv_b    = conv_block1.conv_block2 + skip + pool1: 64 N in + 64 N out + 12 N skip input + 4 N rowptr + 8 E
    #   flops     : algorithmic (LUT form) 2*E*Cin*Cout + 2*N*(root + skip); executed (slot form) counts the 15-slot phases
    kernels = {
        "l1_build": dict(kernel="k_l1_build (+ k_l1_build_dense): spiral radius-graph probe on a shared-memory hashed grid fused with "
                                "SplineConv 3->16 + BN + act", bytes=96 * N + 24 * E,
                         flops_algorithmic=2.0 * (E * 48 + N * 48), flops_executed=2.0 * (E * 45 + N * (15 * 48 + 48)), ncu="k_l1_build"),
        "l1_conv_b_pool_voxel": dict(kernel="k_l1_conv_b2 (+ k_l1_conv_b2_dense): fused SplineConv 16->16 + BN + skip + act + pool1 max/mean/round, "
                                            "TMA-staged, one CTA per voxel", bytes=N * (64 + 64 + 12 + 4) + 8 * E,
                                     flops_algorithmic=2.0 * (E * 256 + N * (256 + 48)), flops_executed=2.0 * (E * 15 * 16 + N * (15 * 256 + 256 + 48)),
                                     ncu="k_l1_conv_b2"),
        "graph_sort": dict(kernel="k_keys_hist + scan + k_scatter + k_rank_emit: cell-major counting sort of the events", bytes=72 * N,
                           flops_algorithmic=0.0, flops_executed=0.0, ncu="graph_sort"),
    }
    entries = []
    for name, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        k = kernels.get(name)
        if k is None or v["ms"] < 0.10 * tot_ms:
            continue
        ach = k["bytes"] / (v["ms"] * 1e-3) / 1e9
        ent = dict(op=name, kernel=k["kernel"], bound="hbm", achieved=ach, peak=peak, unit="GB/s", frac=ach / peak,
                   traffic=(ncu_traffic.get(k["ncu"]) or {}).get("dram_bytes"), peak_source=peak_src,
                   algorithmic_bytes_per_launch=int(k["bytes"]), launch_ms=v["ms"], share_of_step=v["ms"] / tot_ms)
        if k["flops_algorithmic"]:
            ent.update(fp32_tflops_algorithmic=k["flops_algorithmic"] / (v["ms"] * 1e-3) / 1e12,
                       fp32_frac_algorithmic=k["flops_algorithmic"] / (v["ms"] * 1e-3) / 1e12 / fp32_peak,
                       fp32_tflops_executed=k["flops_executed"] / (v["ms"] * 1e-3) / 1e12,
                       fp32_frac_executed=k["flops_executed"] / (v["ms"] * 1e-3) / 1e12 / fp32_peak, fp32_peak_tflops=fp32_peak)
        entries.append(ent)
    step_bytes = N * 320 + 40 * E                                       # SURVEY 8(d): 320 + 40 d bytes per event
    roofline = dict(entries[0]) if entries else {}
    roofline.update(kernels=entries, mean_degree=E / max(N, 1), step_algorithmic_bytes=int(step_bytes),
                    step_frac=step_bytes / (ms * 1e-3) / 1e9 / peak,
                    fp32_peak_source="148 SMs x 4 SMSPs x 32 lanes x 2 FMA (packed FFMA2) x 2 flop, one warp instruction per 2 cycles per SMSP "
                                     "(profiles/r01_ubench_pipes.txt), at the SM clock sampled during the run",
                    note="`roofline` is the kernel with the largest share of the step; `kernels` lists every kernel >= 10 % of the step; "
                         "traffic = DRAM bytes per launch from the committed ncu capture (profiles/ncu_traffic.json), not measured in this run",
                    per_op_ms={k: round(v["ms"], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])})

    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=warm, ms_per_step=ms,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", config=config,
                e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roofline, serial_ms_per_step=serial_ms)
    if sustained is not None:
        line["sustained"] = sustained

    if not a.headline_only:
        # ---- the clustered stream beside the uniform one (SURVEY 8d: "uniform and clustered") ----------------------
        other = "clustered" if a.kind == "uniform" else "uniform"
        del dev_in
        m2, _, _, nev2, step2 = make_workload(a.size, other, 42 + 1000 * 2)
        m2.engine.overlap = not a.no_overlap
        ms2, _, _ = timed(m2.engine, step2, a.steps, warm)
        m2.engine.overlap = False
        prof2, N2, E2 = per_op(m2, step2, min(a.steps, 10))
        line[other] = dict(value=nev2 * world / (ms2 * 1e-3) / 1e6, unit=UNIT, ms_per_step=ms2, mean_degree=E2 / max(N2, 1),
                           per_op_ms={k: round(v["ms"], 4) for k, v in sorted(prof2.items(), key=lambda kv: -kv[1]["ms"])[:6]},
                           note=f"same model / batch / loop as the headline on the {other} stream")
        del m2, step2
        torch.cuda.empty_cache()
        # ---- config 4 (dagr-m, batch 8 per GPU, detections all-gathered) when sharded -------------------------------
        if world > 1:
            m4, _, _, nev4, step4 = make_workload("m", a.kind, 42 + 1000 * 4)
            m4.engine.overlap = not a.no_overlap
            ms4, _, _ = timed(m4.engine, step4, a.steps, warm)
            line.setdefault("extra", {})["config4"] = dict(model="dagr-m", global_batch=a.batch * world, value=nev4 * world / (ms4 * 1e-3) / 1e6,
                                                           unit=UNIT, ms_per_step=ms4, n_gpus=world)
            del m4, step4
            torch.cuda.empty_cache()
        # ---- config 5: every rank runs its own stream at the same time (one stream per GPU, "replicas"); config 3: rank 0 ---
        try:
            mine = measure_streaming(a, dev)
        except Exception as e:                                       # pragma: no cover
            mine = dict(error=repr(e))
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            ok = [g for g in gathered if "error" not in g]
            mine = dict(ok[0]) if ok else dict(gathered[0])
            if ok:
                mine.update(streams=len(ok), aggregate_sustained_mev_s=sum(g["sustained_mev_s"] for g in ok),
                            latency_ms_per_rank=[g["latency_ms"] for g in ok], realtime=all(g["realtime"] for g in ok),
                            note=ok[0]["note"] + f"; {len(ok)} independent streams, one per GPU, measured concurrently")
        line["streaming"] = mine
        if rank == 0:
            try:
                line["interframe_latency_ms"] = measure_interframe(a, dev)
            except Exception as e:                                   # pragma: no cover
                line["interframe_latency_ms"] = dict(error=repr(e))
        barrier()
    sampler.stop_flag = True

    # ---- CPU baseline beside it (rank 0, N = 1 only) ---------------------------------------------
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        sd = {k: v.cpu() for k, v in model.state_dict().items()}
        cal = cpu_calibrate(sd, margs, raws[0])
        threads = cal["threads"]
        n_target = int(min(a.events, max(2000, cal["events"] * (a.cpu_seconds / 2) / max(cal["sec_per_step"], 1e-3))))
        r = cpu_reference_run(sd, margs, raws[0], n_target, 2, 0, threads)
        line["cpu_baseline"] = dict(value=r["mev_s"], unit=UNIT, cores=threads, kind="port", sample=r["sample"])
    if dumped is not None:
        import numpy as np
        out = Path(a.dump_outputs)
        out.mkdir(parents=True, exist_ok=True)
        for name, arr in dumped.items():
            np.save(out / f"{name}.npy", arr)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
