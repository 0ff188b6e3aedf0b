#!/usr/bin/env python
"""ORACLE tooling — generate tests/golden/*.npz by running the UNMODIFIED reference modules.

Needs a checkout of the reference project (basic-pitch).  The reference's third-party imports are
satisfied by oracle/ref_shims (librosa / pretty_midi / mir_eval / resampy stand-ins, and an
`onnxruntime` stand-in whose arithmetic is oracle/model_ref.py), so every line of the reference's
`inference.py` host logic and `note_creation.py` decode executes as shipped.

    python oracle/make_golden.py REFERENCE_CHECKOUT     # rewrites tests/golden/

Fixtures written (all committed, every file < 1 MB):
  vocadito10_pcm44k.npz the same clip as stored in the reference's test resources (44.1 kHz int16 mono): ingest tests
  vocadito10.npz        reference golden note/onset posteriorgrams and events (tests/resources/vocadito_10/*.npz),
                        the events the reference decode emits for the golden posteriorgrams under several
                        parameter sets, and every 64th sample of the 22 050 Hz audio they are checked with
                        (the tests rebuild that audio from vocadito10_pcm44k.npz)
  vocadito10_contour.npz  reference golden contour posteriorgram
  decode_cases/*.npz    posteriorgram inputs (uint16-quantised) + reference decode outputs, one file per group
  host_cases.npz        window counts / unwrap lengths from the reference's windowing code
  predict_2s.npz        config-1 clip: int16 audio + reference predict() outputs (fake-ORT oracle model)
"""
import hashlib
import io
import pathlib
import sys
import tempfile
import warnings

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = pathlib.Path(sys.argv[1]).resolve()
sys.path[:0] = [str(ROOT / "oracle" / "ref_shims"), str(REF), str(ROOT)]

import basic_pitch  # noqa: E402  (the reference package)

assert str(REF) in basic_pitch.__file__, basic_pitch.__file__
from basic_pitch import inference as ref_inf  # noqa: E402
from basic_pitch import note_creation as ref_nc  # noqa: E402

from basic_pitch_b200 import synth, weights  # noqa: E402
from oracle import model_ref, host_ref  # noqa: E402

GOLD = ROOT / "tests" / "golden"
ONNX = REF / "basic_pitch/saved_models/icassp_2022/nmp.onnx"
RES = REF / "tests/resources"


def quant(a: np.ndarray) -> np.ndarray:
    return np.clip(np.round(a.astype(np.float64) * 65535.0), 0, 65535).astype(np.uint16)


def dequant(q: np.ndarray) -> np.ndarray:
    return q.astype(np.float32) / np.float32(65535.0)


def pack_events(events):
    """events: list of (start, end, pitch, amp, bends|None) -> dict of arrays."""
    n = len(events)
    starts = np.array([e[0] for e in events], dtype=np.float64).reshape(n)
    ends = np.array([e[1] for e in events], dtype=np.float64).reshape(n)
    pitch = np.array([e[2] for e in events], dtype=np.int32).reshape(n)
    amp = np.array([e[3] for e in events], dtype=np.float32).reshape(n)
    off = [0]
    flat = []
    has = np.zeros(n, dtype=np.uint8)
    for i, e in enumerate(events):
        b = e[4] if len(e) > 4 else None
        if b is not None:
            has[i] = 1
            flat.extend(int(v) for v in b)
        off.append(len(flat))
    return {
        "start": starts,
        "end": ends,
        "pitch": pitch,
        "amp": amp,
        "bend_flat": np.array(flat, dtype=np.int32),
        "bend_off": np.array(off, dtype=np.int32),
        "bend_has": has,
    }


def ref_decode(post, **kw):
    """Run the reference decode on copies (it mutates its inputs in place)."""
    out = {k: np.array(v, copy=True) for k, v in post.items()}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        frames_notes = ref_nc.output_to_notes_polyphonic(
            np.array(out["note"], copy=True),
            np.array(out["onset"], copy=True),
            onset_thresh=kw.get("onset_thresh", 0.5),
            frame_thresh=kw.get("frame_thresh", 0.3),
            infer_onsets=kw.get("infer_onsets", True),
            min_note_len=kw.get("min_note_len", 11),
            min_freq=kw.get("min_freq"),
            max_freq=kw.get("max_freq"),
            melodia_trick=kw.get("melodia_trick", True),
        )
        _midi, events = ref_nc.model_output_to_notes(
            out,
            onset_thresh=kw.get("onset_thresh", 0.5),
            frame_thresh=kw.get("frame_thresh", 0.3),
            infer_onsets=kw.get("infer_onsets", True),
            min_note_len=kw.get("min_note_len", 11),
            min_freq=kw.get("min_freq"),
            max_freq=kw.get("max_freq"),
            include_pitch_bends=True,
            multiple_pitch_bends=kw.get("multiple_pitch_bends", False),
            melodia_trick=kw.get("melodia_trick", True),
        )
    fr = np.array([[a, b, p] for a, b, p, _ in frames_notes], dtype=np.int32).reshape(-1, 3)
    return fr, events


PARAM_SETS = [
    dict(),
    dict(onset_thresh=0.3, frame_thresh=0.3, min_note_len=5),
    dict(onset_thresh=0.8, frame_thresh=0.1),
    dict(onset_thresh=0.5, frame_thresh=0.0),
    dict(onset_thresh=0.0, frame_thresh=0.5),
    dict(melodia_trick=False),
    dict(infer_onsets=False),
    dict(min_freq=110.0, max_freq=880.0),
    dict(onset_thresh=0.6, frame_thresh=0.4, min_note_len=20, melodia_trick=True, max_freq=2000.0),
]


def add_case(store, name, post, params):
    fr, events = ref_decode(post, **params)
    pe = pack_events(events)
    store[f"{name}/frames"] = fr
    for k, v in pe.items():
        store[f"{name}/{k}"] = v
    store[f"{name}/params"] = np.array(
        [
            params.get("onset_thresh", 0.5),
            params.get("frame_thresh", 0.3),
            params.get("min_note_len", 11),
            1.0 if params.get("infer_onsets", True) else 0.0,
            1.0 if params.get("melodia_trick", True) else 0.0,
            params["min_freq"] if params.get("min_freq") is not None else -1.0,
            params["max_freq"] if params.get("max_freq") is not None else -1.0,
        ],
        dtype=np.float64,
    )
    return len(events)


def smooth_fuzz(rng, n_t, n_f, density):
    """Blobby random activations in [0,1]: sparse impulses smoothed along time."""
    a = (rng.random((n_t + 40, n_f)) < density / 20.0).astype(np.float64) * rng.random((n_t + 40, n_f))
    k = np.exp(-np.arange(40) / rng.uniform(4, 12))
    out = np.zeros((n_t, n_f))
    for f in range(n_f):
        out[:, f] = np.convolve(a[:, f], k)[40 : 40 + n_t]
    out += 0.05 * rng.random((n_t, n_f))
    return np.clip(out, 0, 1).astype(np.float32)


def main() -> None:
    GOLD.mkdir(parents=True, exist_ok=True)
    w = weights.extract_from_onnx(ONNX)

    # ---------------------------------------------------------------- A. vocadito golden
    import librosa  # the shim

    wav = RES / "vocadito_10.wav"
    audio22k, _ = librosa.load(str(wav), sr=22050, mono=True)
    gold_out = np.load(RES / "vocadito_10/model_output.npz", allow_pickle=True)["arr_0"].item()
    gold_ev = np.load(RES / "vocadito_10/note_events.npz", allow_pickle=True)["arr_0"]
    model = ref_inf.Model(ONNX)
    assert model.model_type == ref_inf.Model.MODEL_TYPES.ONNX
    out, _midi, events = ref_inf.predict(str(wav), model)
    for k in ("note", "onset", "contour"):
        assert out[k].shape == gold_out[k].shape, (k, out[k].shape)
        print(f"reference predict() via oracle model vs golden {k}: max-abs {np.abs(out[k] - gold_out[k]).max():.3e}")
    print(f"events: reference-run {len(events)}  golden {len(gold_ev)}")
    store = {
        "audio22k_every64": audio22k.astype(np.float32)[::64].copy(),
        "gold_note": gold_out["note"].astype(np.float32),
        "gold_onset": gold_out["onset"].astype(np.float32),
    }
    for k, v in pack_events([tuple(r) for r in gold_ev]).items():
        store[f"gold_events/{k}"] = v
    post = {k: gold_out[k] for k in ("note", "onset", "contour")}
    for i, p in enumerate(PARAM_SETS):
        n = add_case(store, f"decode{i}", post, p)
        print(f"  vocadito decode{i} {p}: {n} events")
    fr0 = store["decode0/frames"]
    assert len(fr0) == len(gold_ev)
    assert np.array_equal(store["decode0/pitch"], store["gold_events/pitch"])
    assert np.array_equal(store["decode0/bend_flat"], store["gold_events/bend_flat"])
    np.savez_compressed(GOLD / "vocadito10.npz", **store)
    np.savez_compressed(GOLD / "vocadito10_contour.npz", gold_contour=gold_out["contour"].astype(np.float32))
    # the clip as stored (44.1 kHz, 16-bit mono): input of the device ingest tests (csrc/ingest.cu)
    from scipy.io import wavfile

    sr44, pcm = wavfile.read(str(wav))
    assert sr44 == 44100 and pcm.dtype == np.int16 and pcm.ndim == 1
    np.savez_compressed(GOLD / "vocadito10_pcm44k.npz", pcm=pcm, sample_rate=np.int32(sr44))

    # ---------------------------------------------------------------- B. decode cases
    store = {}
    names = []
    rng = np.random.default_rng(1234)

    def add_post(name, post, param_sets):
        q = {k: quant(post[k]) for k in ("note", "onset", "contour")}
        dq = {k: dequant(v) for k, v in q.items()}
        for k, v in q.items():
            store[f"{name}/{k}_q"] = v
        for i, p in enumerate(param_sets):
            n = add_case(store, f"{name}/p{i}", dq, p)
            names.append(f"{name}/p{i}")
            print(f"  {name}/p{i} {p}: {n} events")

    clip = synth.random_notes_clip(10.0, seed=3)
    win = host_ref.window_audio(clip)
    o = model_ref.forward_batched(win, w)
    post = {k: host_ref.unwrap(o[k], len(clip)) for k in o}
    add_post("notes10s", post, PARAM_SETS)

    clip = synth.dense_chords_clip(4.0, seed=7)
    win = host_ref.window_audio(clip)
    o = model_ref.forward_batched(win, w)
    post = {k: host_ref.unwrap(o[k], len(clip)) for k in o}
    add_post("chords4s", post, PARAM_SETS[:4])

    for j, (n_t, dens) in enumerate([(300, 0.3), (257, 1.0), (64, 2.0)]):
        post = {
            "note": smooth_fuzz(rng, n_t, 88, dens),
            "onset": smooth_fuzz(rng, n_t, 88, dens * 0.5),
            "contour": smooth_fuzz(rng, n_t, 264, dens),
        }
        add_post(f"fuzz{j}", post, PARAM_SETS[:6])

    # silence-like: constant in time -> max(frame_diff) == 0 -> NaN path (SURVEY Appendix B.2)
    post = {
        "note": np.full((200, 88), 0.12, np.float32),
        "onset": np.full((200, 88), 0.05, np.float32),
        "contour": np.full((200, 264), 0.1, np.float32),
    }
    add_post("constant", post, [dict(), dict(onset_thresh=0.0, frame_thresh=0.1), dict(frame_thresh=0.1, infer_onsets=False)])

    for n_t in (1, 2, 3, 12, 13, 25):
        post = {
            "note": smooth_fuzz(rng, n_t, 88, 3.0),
            "onset": smooth_fuzz(rng, n_t, 88, 3.0),
            "contour": smooth_fuzz(rng, n_t, 264, 3.0),
        }
        add_post(f"tiny{n_t}", post, [dict(), dict(onset_thresh=0.0, frame_thresh=0.05, min_note_len=1)])
    (GOLD / "decode_cases").mkdir(exist_ok=True)
    groups = {"notes10s": ("notes10s",), "chords4s": ("chords4s",), "fuzz": ("fuzz0", "fuzz1", "fuzz2"),
              "short": ("constant", "tiny1", "tiny2", "tiny3", "tiny12", "tiny13", "tiny25")}
    for group, bases in groups.items():  # tests/golden_util.DECODE_CASE_GROUPS
        part = {k: v for k, v in store.items() if k.split("/")[0] in bases}
        part["names"] = np.array([n for n in names if n.split("/")[0] in bases])
        np.savez_compressed(GOLD / "decode_cases" / f"{group}.npz", **part)

    # ---------------------------------------------------------------- C. host logic
    lens = [1, 3840, 36163, 36164, 36165, 40004, 44100, 72328, 72329, 200607, 220500, 3969000]
    n_windows, n_frames = [], []
    hop = ref_inf.AUDIO_N_SAMPLES - 30 * ref_inf.FFT_HOP
    for n in lens:
        x = np.concatenate([np.zeros(3840, np.float32), np.zeros(n, np.float32)])
        nw = sum(1 for _ in ref_inf.window_audio_file(x, hop))
        fake = np.zeros((nw, 172, 2), np.float32)
        u = ref_inf.unwrap_output(fake, n, 30, hop)
        n_windows.append(nw)
        n_frames.append(u.shape[0])
    # content check on one ragged length
    x = np.arange(100000, dtype=np.float32) / 100000.0
    xw = np.concatenate([np.zeros(3840, np.float32), x])
    wins = np.concatenate([wd[None, :, 0] for wd, _ in ref_inf.window_audio_file(xw, hop)])
    np.savez_compressed(
        GOLD / "host_cases.npz",
        lens=np.array(lens),
        n_windows=np.array(n_windows),
        n_frames=np.array(n_frames),
        ramp_windows_sha=np.frombuffer(hashlib.sha256(wins.tobytes()).digest(), dtype=np.uint8),
        ramp_n_windows=np.array(wins.shape[0]),
    )
    print("host cases:", dict(zip(lens, zip(n_windows, n_frames))))

    # ---------------------------------------------------------------- D. config 1 through reference predict()
    from scipy.io import wavfile

    clip = synth.tones_clip(2.0, seed=0)
    pcm = np.clip(np.round(clip * 32767.0), -32768, 32767).astype(np.int16)
    with tempfile.TemporaryDirectory() as tmp:
        wav = pathlib.Path(tmp) / "cfg1.wav"
        wavfile.write(wav, 22050, pcm)
        out, _midi, events = ref_inf.predict(str(wav), model)
    store = {"pcm16": pcm, "note": out["note"], "onset": out["onset"], "contour": out["contour"]}
    for k, v in pack_events(events).items():
        store[f"events/{k}"] = v
    print(f"config-1 clip: {out['note'].shape[0]} frames, {len(events)} events")
    np.savez_compressed(GOLD / "predict_2s.npz", **store)

    for f in sorted(GOLD.glob("**/*.npz")):
        print(f"{f.name}: {f.stat().st_size} B")


if __name__ == "__main__":
    main()
