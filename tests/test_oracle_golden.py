"""Pin the oracle (CPU restatement) against the reference's own golden vectors and against outputs of
the unmodified reference modules (fixtures made by oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest

from oracle import decode_ref, host_ref, model_ref
from tests.golden_util import (assert_events_equal, case_expected, case_params, dequant, events_to_arrays,
                               load_decode_cases, load_vocadito)


def test_model_restatement_vs_reference_golden(golden_dir, weights_np):
    """reference: tests/test_inference.py:66-70 checks every runtime against this vector at atol=1e-4.
    Here the 44.1 kHz -> 22.05 kHz resampler differs from librosa's soxr_hq, which costs ~2e-4
    (measured 4.6e-5 / 2.1e-4 / 1.1e-4); tolerance 5e-4."""
    z = load_vocadito(golden_dir)
    audio = z["audio22k"]
    assert audio.shape[0] == 200607  # reference: tests/test_inference.py:194
    win = host_ref.window_audio(audio)
    assert win.shape == (6, 43844)  # reference: tests/test_inference.py:164-180
    out = model_ref.forward(win, weights_np)
    for k in ("note", "onset", "contour"):
        got = host_ref.unwrap(out[k], audio.shape[0])
        gold = z[f"gold_{k}"]
        assert got.shape == gold.shape
        assert np.abs(got - gold).max() < 5e-4, k


def test_model_restatement_f32_vs_f64(golden_dir, weights_np):
    import torch

    z = load_vocadito(golden_dir)
    win = host_ref.window_audio(z["audio22k"])[:2]
    a = model_ref.forward(win, weights_np, torch.float32)
    b = model_ref.forward(win, weights_np, torch.float64)
    for k in a:
        assert np.abs(a[k] - b[k]).max() < 1e-4, k


def _run_decode(post, params):
    post = {k: np.array(v, copy=True) for k, v in post.items()}
    with np.errstate(all="ignore"):
        wb, ev = decode_ref.model_output_to_note_events(
            post,
            onset_thresh=params["onset_thresh"],
            frame_thresh=params["frame_thresh"],
            infer_onsets_flag=params["infer_onsets"],
            min_note_len=params["min_note_len"],
            min_freq=params["min_freq"],
            max_freq=params["max_freq"],
            melodia_trick=params["melodia_trick"],
        )
    return events_to_arrays(wb, ev)


def test_decode_restatement_vs_reference_golden_events(golden_dir):
    """reference: tests/test_inference.py:72-76 (28 golden events)."""
    z = load_vocadito(golden_dir)
    post = {k: z[f"gold_{k}"] for k in ("note", "onset", "contour")}
    got = _run_decode(post, dict(onset_thresh=0.5, frame_thresh=0.3, min_note_len=11, infer_onsets=True,
                                 melodia_trick=True, min_freq=None, max_freq=None))
    exp = {k: z[f"gold_events/{k}"] for k in ("start", "end", "pitch", "amp", "bend_flat", "bend_off")}
    assert len(got["pitch"]) == 28
    np.testing.assert_array_equal(got["pitch"], exp["pitch"])
    np.testing.assert_array_equal(got["bend_flat"], exp["bend_flat"])
    np.testing.assert_allclose(got["start"], exp["start"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["end"], exp["end"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["amp"], exp["amp"], rtol=0, atol=1e-5)  # golden was made by another runtime


@pytest.mark.parametrize("i", range(9))
def test_decode_restatement_vs_reference_run_vocadito(golden_dir, i):
    z = load_vocadito(golden_dir)
    post = {k: z[f"gold_{k}"] for k in ("note", "onset", "contour")}
    got = _run_decode(post, case_params(z, f"decode{i}"))
    assert_events_equal(got, case_expected(z, f"decode{i}"), ctx=f"decode{i}")


def test_decode_restatement_vs_reference_run_cases(golden_dir):
    z = load_decode_cases(golden_dir)
    for name in z["names"]:
        name = str(name)
        base = name.rsplit("/", 1)[0]
        post = {k: dequant(z[f"{base}/{k}_q"]) for k in ("note", "onset", "contour")}
        got = _run_decode(post, case_params(z, name))
        assert_events_equal(got, case_expected(z, name), ctx=name)


def test_host_restatement_vs_reference(golden_dir):
    import hashlib

    z = np.load(golden_dir / "host_cases.npz")
    for n, nw, nf in zip(z["lens"], z["n_windows"], z["n_frames"]):
        if n > 400000:
            continue
        win = host_ref.window_audio(np.zeros(int(n), np.float32))
        assert win.shape[0] == nw, n
        assert host_ref.unwrap(np.zeros((win.shape[0], 172, 2), np.float32), int(n)).shape[0] == nf, n
    ramp = np.arange(100000, dtype=np.float32) / 100000.0
    wins = host_ref.window_audio(ramp)
    assert wins.shape[0] == int(z["ramp_n_windows"])
    assert hashlib.sha256(wins.tobytes()).digest() == z["ramp_windows_sha"].tobytes()
