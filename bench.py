#!/usr/bin/env python
"""bench.py - alignments/sec of the ffsubsync hot path on B200 (BASELINE.json metric).

A "step" = one pass of the whole hot path (VAD on 2 h of 16 kHz PCM -> K=5 ratio candidates
rasterised -> windowed FFT correlation + exact re-score -> max over ratios) over one batch of
synthetic pairs per GPU.  `value` counts whole-job alignments (pairs) per second with the PCM
already resident in HBM; `e2e` is the same call through the C ABI with HOST (pinned) buffers,
H2D/D2H inside the timed region.  `--impl reference` times the reference's own CPU algorithm
(numpy complex128 FFT aligner + the numpy restatement of the detector, oracle/) on the host
cores of the same box.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs /tmp/b200_outputs
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 5 --warmup 3
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

METRIC = "alignments/sec (2h@100Hz signals)"
UNIT = "alignments/s"
DURATION_S = 7200.0
FRAME_RATE = 16000
FPW = 160
SAMPLE_RATE = 100
MAX_OFFSET_SECONDS = 60
# SURVEY.md section 8d: compulsory bytes per 2 h pair
BYTES_VAD = 2 * FRAME_RATE * int(DURATION_S) + 4 * SAMPLE_RATE * int(DURATION_S)   # 233 280 000


def bytes_align(k):
    return 4 * 720000 * (1 + k) + 8 * k


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy bandwidth)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml_samples, self.nvml_stop, self.nvml_thread = None, None, None

    def _start_nvml(self):
        """Poll NVML every ~2 ms from a thread (the timed region can be shorter than one
        nvidia-smi sampling period)."""
        import pynvml
        pynvml.nvmlInit()
        dev = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(dev, pynvml.NVML_CLOCK_SM)
        self.nvml_samples, self.nvml_stop = [], threading.Event()
        names = {"hw_slowdown": pynvml.nvmlClocksEventReasonHwSlowdown,
                 "hw_thermal_slowdown": pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": pynvml.nvmlClocksEventReasonSwThermalSlowdown,
                 "sw_power_cap": pynvml.nvmlClocksEventReasonSwPowerCap}

        def loop():
            while not self.nvml_stop.is_set():
                clk = pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM)
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(dev)
                self.nvml_samples.append((clk, [n for n, bit in names.items() if mask & bit]))
                time.sleep(0.002)

        self.nvml_thread = threading.Thread(target=loop, daemon=True)
        self.nvml_thread.start()

    def start(self):
        try:
            self._start_nvml()
            return
        except Exception:
            self.nvml_samples = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml_samples is not None:
            self.nvml_stop.set()
            self.nvml_thread.join(1.0)
            clocks = [c for c, _ in self.nvml_samples]
            reasons = sorted({r for _, rs in self.nvml_samples for r in rs})
            return {"sm_mhz": float(np.median(clocks)) if clocks else None,
                    "sm_min_mhz": float(min(clocks)) if clocks else None, "sm_max_mhz": float(self.sm_max),
                    "samples": len(clocks), "reasons": reasons, "source": "nvml, sampled during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for row in self.rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [c for c in sm if c > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None,
                "sm_max_mhz": max(smax) if smax else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------ GPU arm

def workload_config(world, B, K):
    """The `config` object both arms print (same keys and values: the reference arm times a bounded
    sample of THIS workload, see its cpu_baseline.sample)."""
    name = ("BASELINE configs[3]: 4096 two-hour pairs sharded over 8 GPUs (512 per GPU)"
            if (world == 8 and B == 512) else
            "BASELINE configs[2]: batch of 256 two-hour pairs per GPU" if B == 256 else
            "batch of %d two-hour pairs per GPU (BASELINE configs[2] workload at another batch size)" % B)
    return {"workload": name + ", with the VAD of configs[1]: 16 kHz mono s16le PCM -> energy/ZCR "
                               "VAD -> MaxScoreAligner over K ratios, max_offset_seconds=60",
            "pairs_per_gpu": B, "ratios": K, "signal_frames": 720000, "pcm_samples_per_pair": 115200000}


def default_pairs(world):
    """BASELINE configs[2]: 256 two-hour pairs on one GPU; configs[3]: 4096 pairs over 8 GPUs =
    512 per GPU.  (2 and 4 GPUs keep 256 per GPU.)  B2_BENCH_PAIRS / --pairs override."""
    env = os.environ.get("B2_BENCH_PAIRS")
    if env:
        return int(env)
    return 512 if world >= 8 else 256


_CHECK_JOBS = []   # filled before the worker pool forks (the PCM of a pair is 230 MB: inherited, not pickled)


def _oracle_check_worker(index):
    """Checker (untimed): one sampled pair through the oracle - numpy detector in 100 s chunks, the
    reference's scaler + rasteriser per ratio, complex128 FFT aligner per ratio, max over ratios."""
    from oracle import aligner_oracle as ao
    from oracle import raster_oracle as ro
    from oracle import vad_oracle as vo
    pcm, starts, ends, ratios = _CHECK_JOBS[index]
    chunk = 2 * FRAME_RATE // SAMPLE_RATE * 10000 // 2
    ref = np.concatenate([vo.energy_zcr_detect(pcm[i:i + chunk], SAMPLE_RATE, FRAME_RATE, 0.0)
                          for i in range(0, len(pcm), chunk)])
    subs = [ro.rasterize(starts, ends, None, SAMPLE_RATE, 0, r)[0] for r in ratios]
    mos = ao.max_offset_samples_of(SAMPLE_RATE, MAX_OFFSET_SECONDS)
    per_ratio, ties = [], 0
    for sub in subs:
        conv = ao.correlation(ref, sub)
        lo, hi = ao.surviving_index_range(len(conv), len(sub), mos)
        idx = lo + int(np.argmax(conv[lo:hi]))
        per_ratio.append((float(conv[idx]), len(conv) - 1 - idx - len(sub)))
        # offsets of this ratio whose score equals the maximum to within the float64 FFT's round-off
        ties += int(np.count_nonzero(conv[lo:hi] >= conv[idx] - 1e-6)) - 1
    k = ao.max_score_select(per_ratio, mos)
    return per_ratio, k, ties


def verify_against_oracle(bs, pairs, pcm_d, pcm_off, ratios, n_sample, seed):
    """Untimed parity check at the benchmarked batch size: the whole batch runs once with the
    per-ratio outputs requested (every ratio re-scored exactly) and once winner-only (the timed
    configuration); a seeded sample of pairs is compared with the oracle ratio by ratio (offset
    exact, score within 1e-5 relative) and the winner triples of both runs must agree."""
    import multiprocessing as mp
    import torch
    B, K = len(pcm_off) - 1, len(ratios)
    dev = pcm_d.device
    all_out = {"score": torch.empty(B * K, dtype=torch.float64, device=dev),
               "offset": torch.empty(B * K, dtype=torch.int32, device=dev)}
    full = bs.sync_device(pcm_d, pcm_off, pairs.cue_start, pairs.cue_end, pairs.cue_off, all_out=all_out)
    torch.cuda.synchronize()
    full = {k: v.cpu().numpy().copy() for k, v in full.items()}
    a_score = all_out["score"].cpu().numpy().reshape(B, K)
    a_off = all_out["offset"].cpu().numpy().reshape(B, K)
    win = bs.sync_device(pcm_d, pcm_off, pairs.cue_start, pairs.cue_end, pairs.cue_off)
    torch.cuda.synchronize()
    win = {k: v.cpu().numpy() for k, v in win.items()}
    same_winner = bool((win["best_offset"] == full["best_offset"]).all()
                       and (win["best_k"] == full["best_k"]).all()
                       and (win["best_score"] == full["best_score"]).all())
    rng = np.random.RandomState(seed)
    sample = sorted(rng.choice(B, size=min(n_sample, B), replace=False).tolist())
    jobs = []
    for b in sample:
        pcm = pcm_d[int(pcm_off[b]):int(pcm_off[b + 1])].cpu().numpy()
        c0, c1 = int(pairs.cue_off[b]), int(pairs.cue_off[b + 1])
        jobs.append((pcm, pairs.cue_start[c0:c1], pairs.cue_end[c0:c1], list(ratios)))
    t0 = time.perf_counter()
    _CHECK_JOBS[:] = jobs
    with mp.get_context("fork").Pool(min(len(jobs), max(1, (os.cpu_count() or 1)))) as pool:
        res = pool.map(_oracle_check_worker, range(len(jobs)), chunksize=1)
    _CHECK_JOBS[:] = []
    bad, max_rel = [], 0.0
    n_ties = sum(r[2] for r in res)
    for b, (per_ratio, k, _) in zip(sample, res):
        for kk, (sc, off) in enumerate(per_ratio):
            rel = abs(a_score[b, kk] - sc) / max(abs(sc), 1.0)
            max_rel = max(max_rel, rel)
            if int(a_off[b, kk]) != int(off) or rel > 1e-5:
                bad.append((b, kk, int(a_off[b, kk]), int(off), float(a_score[b, kk]), float(sc)))
        sc, off = per_ratio[k]
        if int(full["best_k"][b]) != k or int(full["best_offset"][b]) != int(off) \
                or abs(full["best_score"][b] - sc) > 1e-5 * max(abs(sc), 1.0):
            bad.append((b, "winner", int(full["best_k"][b]), k, int(full["best_offset"][b]), int(off)))
    return {"ok": (not bad) and same_winner, "pairs_checked": sample, "ratios_checked": K,
            "winner_only_equals_all_ratios": same_winner, "max_score_rel_err": max_rel,
            "exact_ties_in_sample": n_ties,
            "mismatches": bad[:8], "oracle_seconds": round(time.perf_counter() - t0, 1),
            "what": "b2_sync_batch on the full batch vs oracle (numpy detector + complex128 FFTAligner + "
                    "MaxScoreAligner) on a seeded sample; offsets exact, scores <= 1e-5 relative"}


def dump_outputs(path, results):
    """Write what the last timed step returned, one float64 .npy per array (int32 offsets and ratio
    indices are exact in float64), so that two builds can be compared output for output.  The inputs
    are seeded, so the same arguments give the same inputs on every run.  24 B per pair: even 8 GPUs x
    512 pairs stay far below 64 MB, so nothing is sampled."""
    os.makedirs(path, exist_ok=True)
    for name, v in results.items():
        np.save(os.path.join(path, name + ".npy"), v.cpu().numpy().astype(np.float64))


def measured_traffic():
    """DRAM bytes per launch of the dominant kernel from this round's `ncu --set full` capture
    (profiles/r2_vad_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep)."""
    p = os.path.join(ROOT, "profiles", "r2_vad_traffic.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh)
    return None


def run_gpu(args):
    import torch
    from ffsubsync_b200 import _native, distributed
    from ffsubsync_b200.batch import BatchSynchronizer
    from ffsubsync_b200.synth import BENCH_RATIOS, make_pairs

    rank, world, local_rank = distributed.init_from_env("nccl")
    numa = distributed.bind_to_gpu_numa(local_rank)   # before any pinned allocation
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ratios = BENCH_RATIOS[: args.ratios] if args.ratios <= len(BENCH_RATIOS) else None
    if ratios is None:
        from ffsubsync_b200.constants import FRAMERATE_RATIOS
        r = np.array(FRAMERATE_RATIOS)
        ratios = [1.0] + list(np.concatenate([r, 1.0 / r]))[: args.ratios - 1]
    K = len(ratios)
    B = args.pairs if args.pairs else default_pairs(world)   # per GPU (weak scaling)
    bs = BatchSynchronizer(ratios, FRAME_RATE, SAMPLE_RATE, 0.0, max_offset_seconds=MAX_OFFSET_SECONDS,
                           device=local_rank)
    h = bs.handle
    # everything (our kernels, torch ops) is ordered on one explicit stream, and that is the stream
    # the timing events are recorded on; the per-step NCCL gather runs on a side stream, ordered
    # after the step's results by an event, so that step i+1 does not wait for it
    stream = torch.cuda.Stream(device=dev)
    side = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    bs.use_torch_stream()

    # ---- synthetic inputs (untimed): masks on the host, PCM synthesised on the device --------
    seeds = [13 + rank * B + b for b in range(B)]
    pairs = make_pairs(seeds, DURATION_S, ratios, handle=h)
    n_win = int(pairs.win_off[-1])
    cls_d = torch.from_numpy(pairs.window_class).to(dev)
    pcm_d = torch.empty(n_win * FPW, dtype=torch.int16, device=dev)
    h.synth_pcm(cls_d.data_ptr(), n_win, FPW, 1234 + rank, out=pcm_d.data_ptr(), memspace=_native.B2_DEVICE)
    del cls_d
    pcm_off = pairs.win_off * FPW
    out = {"best_score": torch.empty(B, dtype=torch.float64, device=dev),
           "best_offset": torch.empty(B, dtype=torch.int32, device=dev),
           "best_k": torch.empty(B, dtype=torch.int32, device=dev)}
    gather = world > 1 and not os.environ.get("B2_BENCH_NO_GATHER")  # the env knob is a diagnostic
    packed = [torch.empty((B, 3), dtype=torch.float64, device=dev) for _ in range(2)]
    packed_ev = [torch.cuda.Event(), torch.cuda.Event()]
    gathered_ev = [None, None]
    state = {"i": 0, "last": None}

    def step():
        # the corpus sits in HBM and nothing rewrites it: B2_DEVICE_RESIDENT lets step i+1's VAD start while
        # step i's last correlation chain is still running (--ordered-calls: plain B2_DEVICE, for A/B)
        bs.sync_device(pcm_d, pcm_off, pairs.cue_start, pairs.cue_end, pairs.cue_off, out=out,
                       inputs_resident=not args.ordered_calls)
        if not gather:
            return
        # the only exchange of the path: per-pair results to rank 0 (NCCL all-gather of 24 B/pair)
        slot = state["i"] & 1
        state["i"] += 1
        if gathered_ev[slot] is not None:
            stream.wait_event(gathered_ev[slot])      # the gather that last read this buffer is done
        p = packed[slot]
        p[:, 0] = out["best_score"]
        p[:, 1] = out["best_offset"].to(torch.float64)
        p[:, 2] = out["best_k"].to(torch.float64)
        packed_ev[slot].record(stream)
        with torch.cuda.stream(side):
            side.wait_event(packed_ev[slot])
            state["last"] = distributed.gather_pair_results(p, B * world, rank, world)
            ev = torch.cuda.Event()
            ev.record(side)
            gathered_ev[slot] = ev

    def drain():   # the caller's stream sees every gather before the end-of-region event
        for ev in gathered_ev:
            if ev is not None:
                stream.wait_event(ev)

    for _ in range(args.warmup):
        step()
    drain()
    torch.cuda.synchronize()
    ok = bool((out["best_offset"].cpu().numpy() == pairs.true_offset).all()
              and (out["best_k"].cpu().numpy() == pairs.true_k).all())

    # ---- timed region ------------------------------------------------------------------------
    # The clock sampler (NVML init + thread start: tens of ms, different on every rank) starts
    # BEFORE the barrier; after the barrier only a stream synchronise separates the ranks from
    # their start events, so no rank records ev0 early and then waits for the others inside
    # its first collective.
    sampler = ClockSampler(local_rank)
    sampler.start()
    steps = args.steps
    launches0 = h.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    stream.synchronize()
    ev0.record(stream)
    t_wall = time.perf_counter()
    done = 0
    while True:
        for _ in range(steps):
            step()
        done += steps
        if not args.min_seconds or world > 1:
            break
        stream.synchronize()
        if time.perf_counter() - t_wall >= args.min_seconds:
            break
    drain()
    ev1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    steps = done
    local_ms = ev0.elapsed_time(ev1)
    elapsed_ms = distributed.max_over_ranks(local_ms, dev)
    launches = h.launch_count - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        if gather:   # the caller on rank 0 receives every rank's pairs: (score, offset, k) columns
            last = state["last"]
            dump_outputs(args.dump_outputs, {"best_score": last[:, 0], "best_offset": last[:, 1],
                                             "best_k": last[:, 2]})
        else:
            dump_outputs(args.dump_outputs, out)
    per_rank = None
    if world > 1:  # every rank's own device time and SM clock, for the record
        mine = torch.tensor([local_ms / steps, float(clocks.get("sm_mhz") or 0.0),
                             float(numa.get("node", -1))], dtype=torch.float64, device=dev)
        allr = torch.empty((world, 3), dtype=torch.float64, device=dev)
        torch.distributed.all_gather_into_tensor(allr, mine)
        ms = allr[:, 0].tolist()
        per_rank = {"ms_per_step": [round(v, 4) for v in ms], "ms_min": round(min(ms), 4),
                    "ms_max": round(max(ms), 4), "spread": round(max(ms) / min(ms) - 1.0, 4),
                    "sm_mhz": allr[:, 1].tolist(), "numa_node": [int(v) for v in allr[:, 2].tolist()]}

    # ---- per-stage device times (CUDA events on the launching stream), rank 0 only -------------
    stages, roofline, e2e, cpu_base, oracle_check = {}, None, None, None, None
    peak, peak_src = measured_peaks()
    if rank == 0:
        ref_off = pairs.win_off
        ref_sig = torch.empty(n_win, dtype=torch.float32, device=dev)

        def timed(fn, reps):
            fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps):
                fn()
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        vad_ms = timed(lambda: h.vad_energy_zcr(pcm_d.data_ptr(), pcm_off, FRAME_RATE, SAMPLE_RATE, 0.0, 100000,
                                                out=ref_sig.data_ptr(), memspace=_native.B2_DEVICE), args.steps)
        lengths = h.rasterize_lengths(pairs.cue_end, pairs.cue_off, ratios, K, False, SAMPLE_RATE)
        sub_off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        sub_sig = torch.empty(int(sub_off[-1]), dtype=torch.float32, device=dev)
        ras_ms = timed(lambda: h.rasterize(pairs.cue_start, pairs.cue_end, None, pairs.cue_off, ratios, K, False,
                                           SAMPLE_RATE, 0.0, out=sub_sig.data_ptr(), out_off=sub_off,
                                           memspace=_native.B2_DEVICE), args.steps)
        sc = torch.empty(B * K, dtype=torch.float64, device=dev)
        of = torch.empty(B * K, dtype=torch.int32, device=dev)
        st = torch.empty(B * K, dtype=torch.int32, device=dev)
        ali_ms = timed(lambda: h.align_batch(ref_sig.data_ptr(), ref_off, sub_sig.data_ptr(), sub_off, B, K,
                                             MAX_OFFSET_SECONDS * SAMPLE_RATE, score=sc.data_ptr(),
                                             offset=of.data_ptr(), status=st.data_ptr(),
                                             memspace=_native.B2_DEVICE), args.steps)
        stages = {"vad_ms": vad_ms, "rasterize_ms": ras_ms, "align_ms": ali_ms}
        achieved = BYTES_VAD * B / (vad_ms * 1e-3) / 1e9
        tr = measured_traffic()
        traffic = traffic_src = None
        if tr:
            ratio = tr["dram_bytes_per_launch"] / float(tr["algorithmic_bytes_per_launch"])
            traffic = BYTES_VAD * B * ratio
            traffic_src = ("ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of a %d-pair launch "
                           "(%s), x%.4f of its algorithmic bytes, scaled to this launch's pairs"
                           % (tr["pairs"], tr["source"], ratio))
        roofline = {"kernel": "vad_lane_kernel<20, 1> (b2_vad_energy_zcr over the whole batch, all SMs)", "bound": "hbm", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src,
                    "frac_note": "the peak is a COPY bandwidth (read+write mix); this kernel is 98.8 %% reads, "
                                 "which HBM3e serves faster than a copy - frac > 1 is not an error. Against the "
                                 "8000 GB/s data-sheet figure: %.3f" % (achieved / 8000.0),
                    "algorithmic_bytes_per_launch": BYTES_VAD * B,
                    "stages_note": "stages_ms time b2_vad_energy_zcr / b2_rasterize / b2_align_batch called "
                                   "one by one; the timed step calls b2_sync_batch, which replaces the float "
                                   "rasteriser by bit masks (no rasterize_ms on that path) and, from 96 pairs on, "
                                   "runs the VAD of sub-batches 2 and 3 on 80 SMs beside the alignment of the "
                                   "previous sub-batch (the step is shorter than vad_ms + align_ms)",
                    "whole_path": {"achieved": (BYTES_VAD + bytes_align(K)) * B * steps
                                   / (elapsed_ms * 1e-3) / 1e9 if world == 1 else None,
                                   "unit": "GB/s (algorithmic bytes of VAD + align over the step time)"}}
        if roofline["whole_path"]["achieved"]:
            roofline["whole_path"]["frac"] = roofline["whole_path"]["achieved"] / peak
        del ref_sig, sub_sig, sc, of, st

        if not args.no_oracle_check:
            oracle_check = verify_against_oracle(bs, pairs, pcm_d, pcm_off, ratios, args.oracle_pairs, 2024 + B)
            ok = ok and oracle_check["ok"]
        if world == 1 and not args.no_cpu_baseline:
            cpu_base = cpu_baseline_sample(K, ratios, budget_pairs=None)

    # ---- e2e: same call, HOST buffers (pinned), H2D + D2H inside the timed region; every rank
    # streams its own shard over its own PCIe link, time = max over ranks ------------------------
    Be = min(args.e2e_pairs, B)
    n_e = int(pairs.win_off[Be]) * FPW
    pcm_h = torch.empty(n_e, dtype=torch.int16, pin_memory=True)
    pcm_h.copy_(pcm_d[:n_e])
    torch.cuda.synchronize()
    cue_hi = int(pairs.cue_off[Be])
    e_args = (pcm_h.numpy(), pcm_off[: Be + 1], pairs.cue_start[:cue_hi], pairs.cue_end[:cue_hi],
              pairs.cue_off[: Be + 1])
    for _ in range(2):
        res = bs.sync_host(*e_args)
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = bs.sync_host(*e_args)   # synchronises before returning: results are on the host
    e_s = distributed.max_over_ranks((time.perf_counter() - t0) / args.steps * 1e3, dev) / 1e3
    ok_e = distributed.max_over_ranks(0.0 if bool((res[1] == pairs.true_offset[:Be]).all()) else 1.0, dev) == 0.0
    ok = ok and ok_e
    h2d = int(n_e * 2 + cue_hi * 16 + (Be + 1) * 16 + K * 8)
    e2e = {"value": Be * world / e_s, "unit": UNIT, "pairs_per_step": Be * world,
           "h2d_bytes_per_step": h2d * world,
           "d2h_bytes_per_step": int(Be * 16) * world, "ms_per_step": e_s * 1e3,
           "h2d_gbs_per_gpu": h2d / e_s / 1e9, "numa": numa,
           "note": "b2_sync_batch with B2_HOST buffers on every rank (own PCIe link each, rank bound to its "
                   "GPU's NUMA node before the pinned allocation), max over ranks; PCIe H2D of the PCM is "
                   "the bound"}
    del pcm_h

    if rank == 0:
        total_pairs = B * world * steps
        line = {
            "metric": METRIC, "value": total_pairs / (elapsed_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64 VAD; f32 FFT nomination + f64 exact re-score", "data": "synthetic",
            "config": dict(workload_config(world, B, K),
                           l2_policy="inputs (%.1f GB PCM per GPU) are far larger than the 126 MB L2" % (B * 0.2304),
                           parallelism="pairs block-sharded, dp%d" % world,
                           call=("b2_sync_batch(B2_DEVICE): every step ordered after the previous one" if args.ordered_calls
                                 else "b2_sync_batch(B2_DEVICE_RESIDENT): the PCM is resident and constant, so the VAD of "
                                      "step i+1 overlaps the last correlation chain of step i; all work of the K steps "
                                      "lies inside the timed region"),
                           exchange=("NCCL all_gather_into_tensor of 24 B/pair per step on a side stream "
                                     "(event-ordered after the step's results)") if gather else None),
            "verified_offsets": ok, "verified_vs_oracle": oracle_check, "gpu_launches": int(launches),
            "clocks": clocks, "per_rank": per_rank, "stages_ms": stages,
            "timed_region_s": elapsed_ms * 1e-3,
            "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu_base,
        }
        print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------------- CPU / reference arm

_CPU_STATE = {}


def _cpu_worker(job):
    """One 2 h pair through the reference's algorithm on one host core: the numpy restatement of
    the detector in 100 s chunks (speech_transformers.py:710-746), the per-ratio scaler +
    rasteriser and the complex128 FFT aligner (aligners.py:50-80), max over ratios."""
    from oracle import aligner_oracle as ao
    from oracle import raster_oracle as ro
    from oracle import vad_oracle as vo
    pcm, starts, ends, ratios = _CPU_STATE["pcm"], _CPU_STATE["starts"], _CPU_STATE["ends"], _CPU_STATE["ratios"]
    chunk = 2 * FRAME_RATE // SAMPLE_RATE * 10000 // 2
    ref = np.concatenate([vo.energy_zcr_detect(pcm[i:i + chunk], SAMPLE_RATE, FRAME_RATE, 0.0)
                          for i in range(0, len(pcm), chunk)])
    subs = [ro.rasterize(starts, ends, None, SAMPLE_RATE, 0, r)[0] for r in ratios]
    (score, off), k = ao.max_score_align(ref, subs, SAMPLE_RATE, MAX_OFFSET_SECONDS)
    return off, k


def _cpu_setup(ratios):
    from oracle import raster_oracle as ro
    from oracle import vad_oracle as vo
    if "pcm" in _CPU_STATE:
        return
    starts, ends = ro.synthetic_cues(13, DURATION_S)
    mask = ro.rasterize(starts, ends, None, SAMPLE_RATE, 0, 1.0)[0] != 0
    n = int(DURATION_S * SAMPLE_RATE)
    ref = np.zeros(n, dtype=bool)
    src = np.arange(n) - 1234
    okm = (src >= 0) & (src < len(mask))
    ref[okm] = mask[src[okm]]
    ref ^= np.random.RandomState(1).rand(n) < 0.10
    _CPU_STATE.update(pcm=vo.synth_pcm(ref.astype(np.uint8), FPW, seed=7), starts=starts, ends=ends,
                      ratios=list(ratios), expect=1234)


def available_cores():
    """Host cores this process may actually use: the container's CPU quota (cgroup v2 cpu.max, v1
    cfs_quota) when there is one, else the affinity mask.  On the bench pod os.cpu_count() says 128
    but cpu.max is "1600000 100000" = 16 cores: 16 workers give 4.9 alignments/s, 32 give 3.1, 128
    give 1.9 (profiles/r2a_cpu_sweep.json) - oversubscribing the quota only adds context switches.
    B2_CPU_WORKERS overrides."""
    if os.environ.get("B2_CPU_WORKERS"):
        return max(1, int(os.environ["B2_CPU_WORKERS"])), "B2_CPU_WORKERS"
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    src = "sched_getaffinity"
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            q = max(1, int(np.ceil(int(quota) / float(period))))
            if q < n:
                n, src = q, "cgroup cpu.max %s/%s" % (quota, period)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as fq, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fp:
                quota, period = int(fq.read()), int(fp.read())
            if quota > 0 and int(np.ceil(quota / period)) < n:
                n, src = int(np.ceil(quota / period)), "cgroup cfs quota"
        except (OSError, ValueError):
            pass
    return max(1, n), src


def cpu_pass(n_pairs, cores):
    import multiprocessing as mp
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_worker(i) for i in range(n_pairs)]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_cpu_worker, range(n_pairs), chunksize=1)
    dt = time.perf_counter() - t0
    assert all(r[0] == _CPU_STATE["expect"] for r in res), res
    return n_pairs / dt, dt


def cpu_baseline_sample(K, ratios, budget_pairs=None):
    for v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[v] = "1"
    cores = os.cpu_count() or 1
    used, quota_src = available_cores()
    _cpu_setup(ratios)
    n_pairs = budget_pairs or used
    rate, dt = cpu_pass(n_pairs, used)
    return {"value": rate, "unit": UNIT, "cores": used, "host_cores": cores, "cores_source": quota_src,
            "kind": "port",
            "sample": "%d two-hour pairs (one per worker process), K=%d ratios, VAD + aligner, %.1f s wall"
                      % (n_pairs, K, dt)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from ffsubsync_b200.synth import BENCH_RATIOS
    ratios = BENCH_RATIOS[: args.ratios]
    K = len(ratios)
    for v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[v] = "1"
    cores = os.cpu_count() or 1
    used, quota_src = available_cores()
    _cpu_setup(ratios)
    per_step = used
    for _ in range(min(args.warmup, 1)):   # one warm-up pass is enough for a CPU pool; bounded runtime
        cpu_pass(per_step, used)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_pass(per_step, used)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64 VAD; complex128 FFT",
        "data": "synthetic",
        "config": dict(workload_config(world, args.pairs if args.pairs else default_pairs(world), K),
                       implementation="the reference's algorithm on the host: energy/ZCR detector (numpy restatement, "
                                      "100 s chunks) -> SubtitleScaler + rasteriser per ratio -> FFTAligner (numpy "
                                      "complex128, aligners.py:50-80) -> MaxScoreAligner",
                       sample_pairs_per_step=per_step),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "host_cores": cores,
                         "cores_source": quota_src, "kind": "port",
                         "sample": "%d two-hour pairs per step, one per worker process" % per_step},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference is pure Python and cannot travel to the GPU box; this is the oracle port of "
                "its algorithm (pinned to the reference by tests/golden) on all host cores",
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=0,
                    help="2 h pairs per GPU per step (default: BASELINE configs[2] = 256 on 1/2/4 GPUs, "
                         "configs[3] = 512 per GPU on 8 GPUs; 59 / 118 GB of PCM per GPU)")
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="1 GPU only: repeat the K timed steps until the timed region is at least this long "
                         "(sustained-clock runs for profiles/; `steps` in the output is what actually ran)")
    ap.add_argument("--oracle-pairs", type=int, default=8,
                    help="pairs of the batch cross-checked against the oracle after the timed region")
    ap.add_argument("--no-oracle-check", action="store_true")
    ap.add_argument("--ratios", type=int, default=5)
    ap.add_argument("--e2e-pairs", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ordered-calls", action="store_true",
                    help="timed steps call b2_sync_batch with B2_DEVICE instead of B2_DEVICE_RESIDENT (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the per-pair results of the last one (best_score, "
                         "best_offset, best_k) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
