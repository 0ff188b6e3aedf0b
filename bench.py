#!/usr/bin/env python
"""Benchmark of the hot path: audio -> HCQT -> CNN -> note events, audio-seconds per second.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                      (CPU baseline arm: the oracle port on host cores)
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's note events as .npy)

Workload (BASELINE.json configs[3], the configuration the 1/2/4/8-GPU metric is quoted on): 10 s synthetic
22 050 Hz clips (every clip its own seed), full pipeline to note events, sharded by file with no data-path
collective.  Weak scaling: every rank transcribes `--clips` (default 1250 = 10 000 / 8) clips per step.  One step =
one pass of the path over that batch.

  value        audio already resident in HBM (bp_transcribe_device), CUDA events, max over ranks
  e2e          the C-ABI host entry point (bp_transcribe_host) from pinned host buffers: H2D of the audio and D2H of
               the note events inside the timed region
  e2e_python   the Python drop-in a user calls: predict_batch(list of unpinned numpy arrays) -> posteriorgrams,
               MIDI objects and note events (packing, H2D, D2H of the posteriorgrams and object assembly included)
  roofline     the dominant tensor-core kernel family of the step (picked from the per-family event timings)
  roofline_decode   stage 3 against the HBM roofline: frames x 1 760 B / decode time (SURVEY.md §8d)
  parity       the oracle run on a fixed sample of THIS step's clips (BASELINE.md §5)
  cpu_baseline the oracle port timed on the host cores (same clips, windows batched across clips)

Inputs per step (1.1 GB) exceed the 126 MB L2, so no explicit L2 flush is needed between iterations.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CLIP_SECONDS = 10.0
SR = 22050
WORKLOAD = "BASELINE configs[3] per-GPU shard: 10 s synthetic 22 050 Hz clips, full pipeline (HCQT+CNN+note decode) to note events, sharded by file"
FLOP_PER_WINDOW = 1_048_159_296  # SURVEY.md §8(d)
DECODE_BYTES_PER_FRAME = 1760  # note + onset + contour rows, fp32 (SURVEY.md §8d)
# kernel families the library can time (bp_model_profile): algorithmic FLOP per window of the tensor-core ones
FAMILIES = {
    0: ("contour conv 8->8 3x39 + fused conv2 8->1 5x5 (conv_tc_kernel<3>, tcgen05 split-bf16, conv2 as TS-form MMAs)", 680_030_208 + 18_163_200),
    1: ("onset conv 8->32 5x5/3 + fused conv2 33->1 3x3 (conv_tc_kernel<1>, tcgen05 split-bf16, conv2 as TS-form MMAs)", 193_740_800 + 8_990_784),
    2: ("constant-Q projection + log-normalise (cqt_tc_kernel, tcgen05 3-way bf16 split)", 57_065_472),
    3: ("decimation chain (FFMA2)", 22_359_552),
    4: ("note conv 1->32 7x7/3 + fused conv2 32->1 7x3 (conv_tc_kernel<2>, tcgen05 split-bf16, conv2 as TS-form MMAs)", 47_466_496 + 20_342_784),
    5: ("decode: prep / candidates / sequential loops", 0),
    6: ("decode: amplitude + pitch bends", 0),
}


def host_threads() -> int:
    """Cores this process may really use (affinity mask and cgroup CPU quota), capped at 32: torch's CPU kernels
    collapse when oversubscribed on a shared host."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()[:2]
            if quota != "max":
                n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 32))


def make_clips(n_clips: int, seed0: int, workers: int = 0):
    """Clip i of a shard is synth.random_notes_clip(10 s, seed0 + i): every clip distinct (SURVEY config 4: seeds 3+i)."""
    from basic_pitch_b200 import synth

    workers = workers or min(16, host_threads())
    if n_clips <= 4 or workers <= 1:
        return [synth.random_notes_clip(CLIP_SECONDS, seed=seed0 + i) for i in range(n_clips)]
    with ThreadPoolExecutor(workers) as ex:  # numpy releases the GIL inside sin/exp
        return list(ex.map(lambda i: synth.random_notes_clip(CLIP_SECONDS, seed=seed0 + i), range(n_clips)))


def workload_config(clips_per_gpu: int, world: int):
    """The part of `config` that both arms (GPU and --impl reference) print identically."""
    n = int(round(CLIP_SECONDS * SR))
    windows = -(-(n + 3840) // 36164)
    frames = int(n / 36164 * 142)
    return {
        "workload": WORKLOAD, "clips_per_gpu_per_step": clips_per_gpu, "clip_seconds": CLIP_SECONDS,
        "clip_seeds": "3 + 100000*rank + i (all clips distinct)", "windows_per_gpu_per_step": windows * clips_per_gpu,
        "frames_per_gpu_per_step": frames * clips_per_gpu, "parallelism": f"files x{world}, no data-path collective",
        "l2": f"inputs {clips_per_gpu * n * 4 / 1e6:.0f} MB per step > 126 MB L2 (no flush needed)",
    }  # fmt: skip


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port
# ---------------------------------------------------------------------------------------------------------------
CPU_GROUP = 19  # clips per model call: 19 x 7 = 133 windows >= 128 per forward (SURVEY probe batched 110)


def cpu_transcribe(clips, w, threads: int):
    """Oracle port over a list of clips: windows of CPU_GROUP clips batched into one torch-CPU forward, decode per
    clip.  Returns (posteriorgrams per clip, frame-indexed notes with bends per clip)."""
    import torch

    from oracle import decode_ref, host_ref, model_ref

    torch.set_num_threads(threads)
    posts, notes = [], []
    for g0 in range(0, len(clips), CPU_GROUP):
        grp = clips[g0 : g0 + CPU_GROUP]
        wins = [host_ref.window_audio(c) for c in grp]
        out = model_ref.forward_batched(np.concatenate(wins), w, batch=160)
        pos = 0
        for c, wn in zip(grp, wins):
            post = {k: host_ref.unwrap(out[k][pos : pos + len(wn)], len(c)) for k in out}
            pos += len(wn)
            with np.errstate(all="ignore"):
                wb, _ev = decode_ref.model_output_to_note_events({k: np.array(v) for k, v in post.items()}, 0.5, 0.3)
            posts.append(post)
            notes.append(wb)
    return posts, notes


def cpu_baseline(n_clips: int, threads: int, seed0: int = 3, repeats: int = 3):
    """The oracle port (torch-CPU fp32 restatement of the deployed graph + NumPy restatement of the reference decode)
    on the host cores, on the first `n_clips` clips of rank 0's shard.  Median of `repeats`.  Returns (audio-s/s, text)."""
    from basic_pitch_b200 import ICASSP_2022_MODEL_PATH, weights

    w = weights.load(ICASSP_2022_MODEL_PATH)
    clips = make_clips(n_clips, seed0)
    times, n_notes = [], 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        _posts, notes = cpu_transcribe(clips, w, threads)
        times.append(time.perf_counter() - t0)
        n_notes = sum(len(x) for x in notes)
    dt = float(np.median(times))
    return n_clips * CLIP_SECONDS / dt, (
        f"first {n_clips} of the step's 10 s clips, windows batched {CPU_GROUP} clips (133 windows) per forward: model "
        f"(torch-CPU fp32, {threads} threads) + decode (NumPy restatement, 1 thread), {n_notes} notes, median of "
        f"{repeats} runs {dt:.2f} s")


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    from basic_pitch_b200 import ICASSP_2022_MODEL_PATH, weights

    threads = host_threads()
    w = weights.load(ICASSP_2022_MODEL_PATH)
    per_step = 2 * CPU_GROUP
    clips = make_clips(per_step, seed0=3)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_transcribe(clips[:CPU_GROUP], w, threads)
    step_s = []
    n_notes = 0
    for _s in range(args.steps):
        t0 = time.perf_counter()
        _posts, notes = cpu_transcribe(clips, w, threads)
        step_s.append(time.perf_counter() - t0)
        n_notes = sum(len(x) for x in notes)
    dt = float(np.sum(step_s))
    value = args.steps * per_step * CLIP_SECONDS / dt
    desc = (f"bounded sample: the first {per_step} of the step's {args.clips} 10 s clips per step, windows batched "
            f"{CPU_GROUP} clips (133 windows) per forward: model (torch-CPU fp32, {threads} threads) + decode (NumPy "
            f"restatement, 1 thread), {n_notes} notes per step, median step {np.median(step_s):.2f} s; restated CPU "
            "baseline (onnxruntime / TensorFlow are not installable offline; the reference's own decode is pure Python "
            "like this port)")
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.clips, world),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# parity of the step's own clips against the oracle (BASELINE.md §5)
# ---------------------------------------------------------------------------------------------------------------
def parity_report(model, clips, sample_idx, threads: int):
    """GPU (public API, same library path as the timed step) vs oracle on clips[sample_idx]."""
    from basic_pitch_b200 import ICASSP_2022_MODEL_PATH, weights
    from oracle import decode_ref

    w = weights.load(ICASSP_2022_MODEL_PATH)
    sample = [clips[i] for i in sample_idx]
    outs, res, _frames = model.transcribe_arrays(sample)
    posts, cpu_notes = cpu_transcribe(sample, w, threads)
    err = {"note": 0.0, "onset": 0.0, "contour": 0.0}
    bit_identical = True
    matched = n_gpu = n_cpu = 0
    for i in range(len(sample)):
        for k in err:
            err[k] = max(err[k], float(np.abs(outs[i][k] - posts[i][k]).max()))
        # (a) the reference decode restated on the CPU, fed the GPU's own posteriorgrams, must give the GPU's note list
        with np.errstate(all="ignore"):
            wb, _ = decode_ref.model_output_to_note_events({k: np.array(v) for k, v in outs[i].items()}, 0.5, 0.3)
        r = res[i]
        got = [(int(a), int(b), int(p), np.float32(x).tobytes(), [int(v) for v in r["bends"][r["bend_off"][j] : r["bend_off"][j + 1]]])
               for j, (a, b, p, x) in enumerate(zip(r["start"], r["end"], r["pitch"], r["amp"]))]
        exp = [(int(a), int(b), int(p), np.float32(x).tobytes(), [int(v) for v in bd]) for a, b, p, x, bd in wb]
        bit_identical = bit_identical and got == exp
        # (b) end to end: CPU oracle on its own posteriorgrams vs the GPU events (start, end, pitch exact)
        g = {(a, b, p) for a, b, p, _x, _bd in got}
        c = {(int(a), int(b), int(p)) for a, b, p, _x, _bd in cpu_notes[i]}
        matched += len(g & c)
        n_gpu += len(g)
        n_cpu += len(c)
    return {
        "sample": f"{len(sample)} clips of this step's batch (indices {list(sample_idx)}), {n_gpu} GPU notes",
        "post_max_abs": err, "post_tolerance": 1e-3,
        "decode_bit_identical_on_gpu_posteriorgrams": bool(bit_identical),
        "e2e_event_agreement": matched / max(1, max(n_gpu, n_cpu)),
        "e2e_events": {"gpu": n_gpu, "cpu_oracle": n_cpu, "identical_start_end_pitch": matched},
    }  # fmt: skip


DUMP_BYTES = 64 << 20  # cap of --dump-outputs


def dump_outputs(dump_dir: str, out) -> None:
    """Write what bp_transcribe_device returned to its caller in the last timed step as dump_dir/<name>.npy: per clip
    `frame_off` and `note_off`, per note `start_frame`, `end_frame`, `pitch_midi`, `amplitude` and `bend_off`, and the
    flat `bends` (offsets as float64, the rest as float32; every integer is exact).  The clips are seeded, so two builds
    given the same arguments can be compared array by array.  Past DUMP_BYTES a fixed seeded sample of whole clips is
    written instead; `clip_index` lists the clips written."""
    a, n_files = out.a, out.n_files
    note_off = a["note_off"][: n_files + 1].astype(np.int64)
    frame_off = a["frame_off"][: n_files + 1].astype(np.int64)
    bend_off = a["bend_off"][: note_off[-1] + 1].astype(np.int64)
    clip_bends = bend_off[note_off]  # bends of clip i: clip_bends[i] .. clip_bends[i + 1]
    cost = 24 + 24 * np.diff(note_off) + 4 * np.diff(clip_bends)  # bytes per clip in the files below
    clips = np.arange(n_files)
    budget = DUMP_BYTES - 4096  # .npy headers and the leading zero of each offset array
    if cost.sum() > budget:
        order = np.random.default_rng(0).permutation(n_files)
        clips = np.sort(order[np.cumsum(cost[order]) <= budget])
    notes = np.concatenate([np.arange(note_off[i], note_off[i + 1]) for i in clips] + [np.zeros(0, np.int64)])

    def rebase(counts):
        return np.concatenate([[0], np.cumsum(counts)]).astype(np.float64)

    arrays = {
        "clip_index": clips.astype(np.float64),
        "frame_off": rebase(np.diff(frame_off)[clips]),
        "note_off": rebase(np.diff(note_off)[clips]),
        "start_frame": a["start"][notes].astype(np.float32),
        "end_frame": a["end"][notes].astype(np.float32),
        "pitch_midi": a["pitch"][notes].astype(np.float32),
        "amplitude": a["amp"][notes].astype(np.float32),
        "bend_off": rebase(np.diff(bend_off)[notes]),
        "bends": np.concatenate([a["bends"][clip_bends[i] : clip_bends[i + 1]] for i in clips] + [np.zeros(0, np.int32)]).astype(np.float32),
    }
    os.makedirs(dump_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(dump_dir, f"{name}.npy"), arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips", type=int, default=1250, help="10 s clips per GPU per step")
    ap.add_argument("--cpu-clips", type=int, default=2 * CPU_GROUP, help="clips of the cpu_baseline sample")
    ap.add_argument("--parity-clips", type=int, default=6, help="clips of the step checked against the oracle")
    ap.add_argument("--python-steps", type=int, default=2, help="timed predict_batch() passes for e2e_python")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the note events of the last timed step to DIR/<name>.npy "
                    "(DIR/rank<r>/ per rank when several ranks run)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    # NCCL prints its version banner on stdout at VERSION/INFO level; the contract is ONE JSON line on stdout
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"

    import torch
    import torch.distributed as dist

    from basic_pitch_b200 import ICASSP_2022_MODEL_PATH, engine
    from basic_pitch_b200.inference import Model, predict_batch

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    model = Model(ICASSP_2022_MODEL_PATH, device=local)
    engine.broadcast_weights(model)  # the one collective of the path

    clips = make_clips(args.clips, seed0=3 + 100000 * rank, workers=max(1, min(16, host_threads() // max(1, min(world, 8)))))
    audio_s = args.clips * CLIP_SECONDS
    packed = engine.PackedAudio(clips, pinned=True)
    lib = model._lib
    n_windows = sum(int(lib.bp_num_windows(len(c))) for c in clips)
    n_frames = sum(int(lib.bp_num_frames(len(c))) for c in clips)
    out = engine.NoteBuffers(args.clips, max(4096, 2 * n_frames), max(65536, 24 * n_frames))
    d_audio = packed.to_device(local)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    dev_step = lambda: engine.transcribe_packed_device(model, d_audio, packed.offsets, out)  # noqa: E731
    host_step = lambda: engine.transcribe_packed_host(model, packed, out)  # noqa: E731

    for _ in range(args.warmup):
        dev_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = model.launch_count
    ms = timed(dev_step, args.steps)
    launches = model.launch_count - l0
    n_notes = out.n_notes()
    if args.dump_outputs:  # before the e2e leg reuses `out`
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), out)
    for _ in range(2):
        host_step()
    ms_e2e = timed(host_step, args.steps)
    d2h = out.result_bytes()
    clocks = sampler.stop() if rank == 0 else None

    # per-family CUDA-event timing (one extra untimed-for-the-metric step per family; events on the launching stream)
    fam = {}
    tot, nint, nwin = C.c_double(), C.c_int64(), C.c_int64()
    for which in FAMILIES:
        lib.bp_model_profile(model.handle, which)
        dev_step()
        lib.bp_model_profile_read(model.handle, C.byref(tot), C.byref(nint), C.byref(nwin))
        fam[which] = {"ms_per_step": tot.value, "launch_groups": int(nint.value), "windows": int(nwin.value)}
    lib.bp_model_profile(model.handle, -1)

    # the Python drop-in: unpinned numpy arrays in, posteriorgrams + MIDI objects + note events out
    py_ms = None
    if args.python_steps > 0:
        res_py = predict_batch(clips, model)  # warm-up: the page-locked output pool is allocated on the first full-size call
        del res_py
        barrier()
        t0 = time.perf_counter()
        res_py = None
        for _ in range(args.python_steps):
            del res_py  # (holding the previous step's posteriorgrams would force a fresh 1.9 GB page-locked allocation)
            res_py = predict_batch(clips, model)
        torch.cuda.synchronize()
        py_s = torch.tensor([(time.perf_counter() - t0) / args.python_steps], device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(py_s, op=dist.ReduceOp.MAX)
        py_ms = 1e3 * float(py_s.item())
        py_d2h = sum(v.nbytes for r in res_py for v in r[0].values())
        del res_py
        barrier()
        # the same call with every note event and MIDI object assembled before it returns (lazy=False)
        t0 = time.perf_counter()
        res_py = predict_batch(clips, model, lazy=False)
        torch.cuda.synchronize()
        py_full_s = torch.tensor([time.perf_counter() - t0], device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(py_full_s, op=dist.ReduceOp.MAX)
        py_full_ms = 1e3 * float(py_full_s.item())
        del res_py
        barrier()

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except OSError:
            pass
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_bw = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained / hbm_gbs)" if peaks else "fallback (B200_PROFILING.md)"
        dom = max((0, 1, 2, 4), key=lambda k: fam[k]["ms_per_step"])
        f_ms, f_groups, f_win = fam[dom]["ms_per_step"], max(1, fam[dom]["launch_groups"]), fam[dom]["windows"]
        achieved = FAMILIES[dom][1] * f_win / (f_ms * 1e-3) / 1e12 if f_ms > 0 else None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
                tj = json.load(fh)
                traffic = tj["families"][str(dom)]["dram_bytes_per_window"] * f_win / f_groups
        except (OSError, KeyError, ValueError, TypeError):
            pass
        # every tensor-core family against the same measured peak (the dominant one is repeated in `roofline`)
        fam_roof = {}
        for k in (0, 1, 2, 4):
            if fam[k]["ms_per_step"] > 0:
                tf = FAMILIES[k][1] * fam[k]["windows"] / (fam[k]["ms_per_step"] * 1e-3) / 1e12
                fam_roof[FAMILIES[k][0].split(" (")[0]] = {
                    "ms_per_step": round(fam[k]["ms_per_step"], 3), "algorithmic_tflops": round(tf, 1), "frac_of_peak": round(tf / peak_tf, 4),
                    "share_of_step": round(fam[k]["ms_per_step"] / (ms / args.steps), 3)}
        dec_ms = fam[5]["ms_per_step"] + fam[6]["ms_per_step"]
        dec_gbs = n_frames * DECODE_BYTES_PER_FRAME / (dec_ms * 1e-3) / 1e9 if dec_ms > 0 else None
        threads = host_threads()
        cpu_v, cpu_desc = cpu_baseline(args.cpu_clips, threads, seed0=3)
        step_idx = sorted({int(round(j * (args.clips - 1) / max(1, args.parity_clips - 1))) for j in range(args.parity_clips)})
        parity = parity_report(model, clips, step_idx, threads)
        value = world * args.steps * audio_s / (ms * 1e-3)
        e2e_v = world * args.steps * audio_s / (ms_e2e * 1e-3)
        line = {
            "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.clips, world),
            "derived": {
                "notes_per_gpu_per_step": n_notes, "windows_per_second_per_gpu": n_windows * args.steps / (ms * 1e-3),
                "us_per_window": 1e3 * ms / args.steps / n_windows,
                "model_flops_fraction_of_peak": n_windows * args.steps * FLOP_PER_WINDOW / (ms * 1e-3) / 1e12 / peak_tf,
                "stage_ms_per_step": {FAMILIES[k][0].split(" (")[0].split(":")[0] + f" [{k}]": round(v["ms_per_step"], 3) for k, v in fam.items()},
            },
            "e2e": {"value": e2e_v, "unit": "audio-s/s", "h2d_bytes_per_step": packed.nbytes, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "api": "bp_transcribe_host (pinned host audio in, note events out)"},
            "e2e_python": None if py_ms is None else {
                "value": world * audio_s / (py_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": py_ms, "frac_of_e2e": (world * audio_s / (py_ms * 1e-3)) / e2e_v,
                "h2d_bytes_per_step": packed.nbytes, "d2h_bytes_per_step": int(py_d2h) + d2h,
                "api": "basic_pitch_b200.inference.predict_batch(list of unpinned float32 numpy arrays) -> (posteriorgrams as views of page-locked arrays, LazyPrettyMIDI, NoteEventList) per clip: bp_transcribe_files_host gathers the arrays itself and streams the posteriorgrams back per sub-batch; host wall clock, max over ranks",
                "passes": args.python_steps,
                "materialized": {"value": world * audio_s / (py_full_ms * 1e-3), "ms_per_step": py_full_ms,
                                 "what": "predict_batch(..., lazy=False): every note event tuple and every Instrument / Note / PitchBend object built before returning (1 pass)"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": FAMILIES[dom][0], "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic,
                         "traffic_unit": "DRAM bytes per launch (ncu, profiles/roofline_traffic.json)", "peak_source": peak_src,
                         "avg_launch_ms": f_ms / f_groups, "windows_per_launch": f_win / f_groups,
                         "flop_per_window": FAMILIES[dom][1]},
            "roofline_families": fam_roof,
            "roofline_decode": {"bound": "hbm", "kernel": "decode_prep + decode_cand + decode_seq + note_finish (decode.cu)",
                                "achieved": dec_gbs, "peak": peak_bw, "unit": "GB/s", "frac": (dec_gbs / peak_bw) if dec_gbs else None,
                                "bytes_per_frame": DECODE_BYTES_PER_FRAME, "frames_per_step": n_frames, "ms_per_step": dec_ms,
                                "note": "stage 3 is a scan plus sequential greedy loops: latency-, not bandwidth-bound"},
            "parity": parity,
            "cpu_baseline": {"value": cpu_v, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": cpu_desc},
        }  # fmt: skip
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
