"""Helpers to read the fixtures written by oracle/make_golden.py."""
import numpy as np

# tests/golden/decode_cases/<group>.npz: one file per group of posteriorgram inputs (every fixture file stays < 1 MB)
DECODE_CASE_GROUPS = ("notes10s", "chords4s", "fuzz", "short")


def dequant(q):
    return q.astype(np.float32) / np.float32(65535.0)


def load_vocadito(golden_dir):
    """The vocadito fixture as one mapping: vocadito10.npz, the golden contour posteriorgram (vocadito10_contour.npz)
    and `audio22k`, the 44.1 kHz clip of vocadito10_pcm44k.npz through the package's host resampler — the same
    samples the reference's golden posteriorgrams were reproduced from, pinned by a stored sample of them."""
    from basic_pitch_b200 import audio_io

    z = dict(np.load(golden_dir / "vocadito10.npz"))
    z.update(np.load(golden_dir / "vocadito10_contour.npz"))
    pcm = np.load(golden_dir / "vocadito10_pcm44k.npz")
    audio = audio_io.resample(pcm["pcm"].astype(np.float32) / np.float32(32768.0), int(pcm["sample_rate"]))
    np.testing.assert_array_equal(audio[::64], z.pop("audio22k_every64"), err_msg="host resampler drifted from the fixture")
    z["audio22k"] = audio
    return z


def load_decode_cases(golden_dir):
    """Every decode case of tests/golden/decode_cases/ as one mapping; "names" lists the cases."""
    cases, names = {}, []
    for group in DECODE_CASE_GROUPS:
        with np.load(golden_dir / "decode_cases" / f"{group}.npz") as z:
            names += [str(n) for n in z["names"]]
            cases.update((k, z[k]) for k in z.files if k != "names")
    cases["names"] = np.array(names)
    return cases


def case_params(z, name):
    p = z[f"{name}/params"]
    return dict(
        onset_thresh=float(p[0]),
        frame_thresh=float(p[1]),
        min_note_len=int(p[2]),
        infer_onsets=bool(p[3]),
        melodia_trick=bool(p[4]),
        min_freq=None if p[5] < 0 else float(p[5]),
        max_freq=None if p[6] < 0 else float(p[6]),
    )


def case_expected(z, name):
    return {k: z[f"{name}/{k}"] for k in ("frames", "start", "end", "pitch", "amp", "bend_flat", "bend_off", "bend_has")}


def events_to_arrays(frames_notes_with_bends, events):
    """Convert decode output lists to the fixture array layout."""
    n = len(events)
    fr = np.array([[a, b, p] for a, b, p, _amp, _bd in frames_notes_with_bends], dtype=np.int32).reshape(-1, 3)
    flat, off = [], [0]
    for e in events:
        if e[4] is not None:
            flat.extend(int(v) for v in e[4])
        off.append(len(flat))
    return {
        "frames": fr,
        "start": np.array([e[0] for e in events], dtype=np.float64).reshape(n),
        "end": np.array([e[1] for e in events], dtype=np.float64).reshape(n),
        "pitch": np.array([e[2] for e in events], dtype=np.int32).reshape(n),
        "amp": np.array([e[3] for e in events], dtype=np.float32).reshape(n),
        "bend_flat": np.array(flat, dtype=np.int32),
        "bend_off": np.array(off, dtype=np.int32),
    }


def assert_events_equal(got, exp, amp_atol=0.0, ctx=""):
    assert got["frames"].shape == exp["frames"].shape, f"{ctx}: {got['frames'].shape[0]} notes, expected {exp['frames'].shape[0]}"
    np.testing.assert_array_equal(got["frames"], exp["frames"], err_msg=f"{ctx}: (start,end,pitch) frames")
    np.testing.assert_array_equal(got["pitch"], exp["pitch"], err_msg=f"{ctx}: pitch")
    np.testing.assert_array_equal(got["start"], exp["start"], err_msg=f"{ctx}: start times")
    np.testing.assert_array_equal(got["end"], exp["end"], err_msg=f"{ctx}: end times")
    np.testing.assert_array_equal(got["bend_off"], exp["bend_off"], err_msg=f"{ctx}: bend offsets")
    np.testing.assert_array_equal(got["bend_flat"], exp["bend_flat"], err_msg=f"{ctx}: pitch bends")
    if amp_atol == 0.0:
        np.testing.assert_array_equal(got["amp"], exp["amp"], err_msg=f"{ctx}: amplitude")
    else:
        np.testing.assert_allclose(got["amp"], exp["amp"], rtol=0, atol=amp_atol, err_msg=f"{ctx}: amplitude")
