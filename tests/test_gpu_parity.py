"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI
(ctypes -> libbp_b200.so), against the oracle and the committed golden fixtures.

Tolerances (floating point, BASELINE.json north_star): posteriorgram max-abs <= 1e-3 vs the reference
model; the FP32 path is expected (and required here) to stay within 1e-4 of the fp32 oracle.
Integer work (note decode) must be bit-identical.
"""
import numpy as np
import pytest

from tests.golden_util import (assert_events_equal, case_expected, case_params, dequant, events_to_arrays,
                               load_decode_cases, load_vocadito)

pytestmark = pytest.mark.gpu

POST_TOL = 1e-4  # vs the fp32 oracle on identical 22 050 Hz input
GOLD_TOL = 5e-4  # vs the reference's golden file (44.1 kHz source, resampler differs; see tests/golden/README.md)


@pytest.fixture(scope="module")
def model():
    from basic_pitch_b200 import ICASSP_2022_MODEL_PATH
    from basic_pitch_b200.inference import Model

    return Model(ICASSP_2022_MODEL_PATH)


def _edge_windows():
    from basic_pitch_b200 import synth

    rng = np.random.default_rng(11)
    w = synth.window_batch(5, seed=2)
    zeros = np.zeros((1, 43844), np.float32)  # exercises divide_no_nan (SURVEY Appendix A.2)
    noise = rng.uniform(-1, 1, (1, 43844)).astype(np.float32)  # full-scale white noise
    tiny = (1e-6 * rng.standard_normal((1, 43844))).astype(np.float32)
    click = np.zeros((1, 43844), np.float32)
    click[0, 20000] = 1.0
    return np.concatenate([w, zeros, noise, tiny, click])


def test_forward_vs_oracle_including_activations(model, weights_np):
    from basic_pitch_b200 import _lib
    from oracle import model_ref

    x = _edge_windows()
    ref = model_ref.forward(x, weights_np, return_intermediates=True)
    lib = _lib.load()
    n = x.shape[0]
    model.set_path(0)  # the FP32 path materialises every activation; the tensor-core path fuses the 32-channel ones away
    try:
        fp32 = model.predict(x[:, :, None])
        for which, key, shape, tol in ((0, "_y", (n, 172, 309), 2e-4), (2, "_n1", (n, 32, 172, 88), 5e-4),
                                       (3, "_o1", (n, 32, 172, 88), 5e-4)):
            buf = np.empty(shape, np.float32)
            lib.bp_debug_activation(model.handle, which, buf.ctypes.data, n)
            err = np.abs(buf - ref[key]).max()
            assert err < tol, f"FP32 path activation {key}: max-abs {err:.3e}"
        for k in ("note", "onset", "contour"):
            assert np.abs(fp32[k] - ref[k]).max() < POST_TOL, f"FP32 path {k}"
    finally:
        model.set_path(1)
    # tensor-core paths: 2 keeps the contour activations (channels-last), 1 (the default) reduces them against the
    # next conv inside the epilogue.  The log-magnitude differs from the fp32 oracle mostly in bins near the 1e-10
    # power floor (split-operand MMA accumulation order); what is held to 1e-4 below are the posteriorgrams
    try:
        model.set_path(2)
        unfused = model.predict(x[:, :, None])
        for which, key, shape, tol in ((0, "_y", (n, 172, 309), 1e-3), (1, "_c1", (n, 8, 172, 264), 2e-3)):
            buf = np.empty(shape, np.float32)
            lib.bp_debug_activation(model.handle, which, buf.ctypes.data, n)
            err = np.abs(buf - ref[key]).max()
            assert err < tol, f"activation {key}: max-abs {err:.3e}"
        for k in ("note", "onset", "contour"):
            assert np.abs(unfused[k] - ref[k]).max() < POST_TOL, f"tensor-core path 2, {k}"
    finally:
        model.set_path(1)
    got = model.predict(x[:, :, None])
    buf = np.empty((n, 172, 309), np.float32)
    lib.bp_debug_activation(model.handle, 0, buf.ctypes.data, n)
    assert np.abs(buf - ref["_y"]).max() < 1e-3
    with pytest.raises(Exception):  # path 1 never materialises the 8-channel image
        lib.bp_debug_activation(model.handle, 1, np.empty((n, 8, 172, 264), np.float32).ctypes.data, n)
    for k in ("note", "onset", "contour"):
        assert got[k].shape == ref[k].shape and got[k].dtype == np.float32
        err = np.abs(got[k] - ref[k]).max()
        assert err < POST_TOL, f"{k}: max-abs {err:.3e}"
    assert np.all(np.isfinite(got["note"])) and np.all(np.isfinite(got["contour"]))


def test_tensor_core_contour_conv_matches_fp32_path(model):
    """tcgen05 path (split-bf16 operands, fp32 accumulate in TMEM) vs the FP32 FFMA kernel of the same layer, on device:
    the activation itself and the three posteriorgrams; includes windows that end in ragged M-tiles (9 and 130 windows)."""
    from basic_pitch_b200 import _lib, synth

    lib = _lib.load()
    for n in (9, 130):
        x = np.concatenate([_edge_windows(), synth.window_batch(n - 9, seed=4)]) if n > 9 else _edge_windows()
        try:
            model.set_path(0)
            ref = model.predict(x)
            c_ref = np.empty((min(n, 128), 8, 172, 264), np.float32)
            if n <= 128:
                lib.bp_debug_activation(model.handle, 1, c_ref.ctypes.data, n)
            model.set_path(2)
            got2 = model.predict(x)
            if n <= 128:
                c_got = np.empty_like(c_ref)
                lib.bp_debug_activation(model.handle, 1, c_got.ctypes.data, n)
                err = np.abs(c_got - c_ref).max()
                assert err < 5e-4, f"contour conv activation: max-abs {err:.3e} (n={n})"
            model.set_path(1)
            got = model.predict(x)
        finally:
            model.set_path(1)
        for k in ref:
            err = np.abs(got[k] - ref[k]).max()
            assert err < 1e-4, f"{k}: tensor-core (fused) vs FP32 path max-abs {err:.3e} (n={n})"
            err = np.abs(got2[k] - ref[k]).max()
            assert err < 1e-4, f"{k}: tensor-core (unfused) vs FP32 path max-abs {err:.3e} (n={n})"


def test_vocadito_golden_posteriorgrams(model, golden_dir, weights_np):
    """reference: tests/test_inference.py:43-70 — shapes, and values vs the golden npz."""
    from oracle import host_ref, model_ref

    z = load_vocadito(golden_dir)
    audio = z["audio22k"]
    out = model.run_inference_arrays([audio])[0]
    o = model_ref.forward(host_ref.window_audio(audio), weights_np)
    for k in ("note", "onset", "contour"):
        gold = z[f"gold_{k}"]
        assert out[k].shape == gold.shape
        assert np.abs(out[k] - gold).max() < GOLD_TOL, k
        assert np.abs(out[k] - host_ref.unwrap(o[k], len(audio))).max() < POST_TOL, k


def _gpu_decode(model, post, p):
    from basic_pitch_b200 import note_creation as nc

    lo, hi = nc.frequency_to_column_range(p["min_freq"], p["max_freq"])
    res = model.decode_arrays([post["note"]], [post["onset"]], [post["contour"]], onset_thresh=p["onset_thresh"],
                              frame_thresh=p["frame_thresh"], min_note_len=p["min_note_len"],
                              infer_onsets=p["infer_onsets"], melodia_trick=p["melodia_trick"], min_pitch_idx=lo,
                              max_pitch_idx=hi)[0]
    ev = nc.note_events_from_arrays(res, post["contour"].shape[0])
    wb = [(int(a), int(b), int(pp), amp, None) for a, b, pp, amp in zip(res["start"], res["end"], res["pitch"], res["amp"])]
    return events_to_arrays(wb, ev)


def test_decode_reference_golden_events(model, golden_dir):
    """reference: tests/test_inference.py:72-76 — the 28 golden events from the golden posteriorgrams."""
    z = load_vocadito(golden_dir)
    post = {k: z[f"gold_{k}"] for k in ("note", "onset", "contour")}
    got = _gpu_decode(model, post, dict(onset_thresh=0.5, frame_thresh=0.3, min_note_len=11, infer_onsets=True,
                                        melodia_trick=True, min_freq=None, max_freq=None))
    assert len(got["pitch"]) == 28
    np.testing.assert_array_equal(got["pitch"], z["gold_events/pitch"])
    np.testing.assert_array_equal(got["bend_flat"], z["gold_events/bend_flat"])
    np.testing.assert_array_equal(got["bend_off"], z["gold_events/bend_off"])
    np.testing.assert_allclose(got["start"], z["gold_events/start"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["end"], z["gold_events/end"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["amp"], z["gold_events/amp"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("i", range(9))
def test_decode_bit_exact_vocadito_param_sets(model, golden_dir, i):
    z = load_vocadito(golden_dir)
    post = {k: z[f"gold_{k}"] for k in ("note", "onset", "contour")}
    got = _gpu_decode(model, post, case_params(z, f"decode{i}"))
    assert_events_equal(got, case_expected(z, f"decode{i}"), ctx=f"decode{i}")


def test_decode_bit_exact_reference_cases(model, golden_dir):
    """Every case produced by the UNMODIFIED reference decode: dense chords, fuzz, thresholds <= 0,
    NaN path (constant input), 1..25-frame inputs, frequency limits, melodia on/off."""
    z = load_decode_cases(golden_dir)
    for name in z["names"]:
        name = str(name)
        base = name.rsplit("/", 1)[0]
        post = {k: dequant(z[f"{base}/{k}_q"]) for k in ("note", "onset", "contour")}
        got = _gpu_decode(model, post, case_params(z, name))
        assert_events_equal(got, case_expected(z, name), ctx=name)


def test_decode_batch_equals_single(model, golden_dir):
    """Files decoded in one batched call give the same events as one call per file (incl. an empty file)."""
    z = load_decode_cases(golden_dir)
    bases = ["notes10s", "fuzz0", "tiny3", "chords4s", "constant"]
    posts = [{k: dequant(z[f"{b}/{k}_q"]) for k in ("note", "onset", "contour")} for b in bases]
    posts.insert(2, {"note": np.zeros((0, 88), np.float32), "onset": np.zeros((0, 88), np.float32), "contour": np.zeros((0, 264), np.float32)})
    batch = model.decode_arrays([p["note"] for p in posts], [p["onset"] for p in posts], [p["contour"] for p in posts])
    for p, b in zip(posts, batch):
        single = model.decode_arrays([p["note"]], [p["onset"]], [p["contour"]])[0]
        for k in single:
            np.testing.assert_array_equal(single[k], b[k], err_msg=k)
    assert len(batch[2]["start"]) == 0


def test_decode_vs_oracle_on_gpu_posteriorgrams(model, weights_np):
    """BASELINE.md §5: GPU note list identical to the reference decode run on the SAME GPU posteriorgrams."""
    from basic_pitch_b200 import synth
    from oracle import decode_ref

    for clip in (synth.random_notes_clip(12.0, seed=21), synth.dense_chords_clip(3.0, seed=7)):
        out = model.run_inference_arrays([clip])[0]
        got = _gpu_decode(model, out, dict(onset_thresh=0.5, frame_thresh=0.3, min_note_len=11, infer_onsets=True,
                                           melodia_trick=True, min_freq=None, max_freq=None))
        with np.errstate(all="ignore"):
            wb, ev = decode_ref.model_output_to_note_events({k: np.array(v) for k, v in out.items()}, 0.5, 0.3)
        assert len(ev) > 5
        assert_events_equal(got, events_to_arrays(wb, ev), ctx="gpu-posteriorgrams")


def test_predict_dropin_config1(model, golden_dir, tmp_path):
    """BASELINE.json configs[0]: one 2 s 22 050 Hz WAV through predict(): plumbing + parity with the
    unmodified reference predict() (fixture predict_2s.npz; its model arithmetic is the oracle's)."""
    from scipy.io import wavfile

    from basic_pitch_b200.inference import predict, predict_and_save

    z = np.load(golden_dir / "predict_2s.npz")
    wav = tmp_path / "cfg1.wav"
    wavfile.write(wav, 22050, z["pcm16"])
    model_output, midi_data, note_events = predict(wav, model)
    assert set(model_output) == {"note", "onset", "contour"}
    for k in ("note", "onset", "contour"):
        assert model_output[k].shape == z[k].shape == (173, 88 if k != "contour" else 264)
        assert np.abs(model_output[k] - z[k]).max() < POST_TOL, k
    assert len(note_events) == len(z["events/pitch"])
    assert [int(e[2]) for e in note_events] == list(z["events/pitch"])
    np.testing.assert_array_equal(np.array([e[0] for e in note_events]), z["events/start"])
    np.testing.assert_array_equal(np.array([e[1] for e in note_events]), z["events/end"])
    flat = [int(b) for e in note_events for b in (e[4] or [])]
    assert sum(abs(a - b) for a, b in zip(flat, z["events/bend_flat"])) <= 2 and len(flat) == len(z["events/bend_flat"])
    assert len(midi_data.instruments) == 1 and len(midi_data.instruments[0].notes) == len(note_events)
    for e in note_events:  # reference: tests/test_inference.py:55-64
        assert 21 <= e[2] <= 108 and e[0] < e[1] <= 2.0 + 2 * 256 / 22050
    out_dir = tmp_path / "out"
    out_dir.mkdir()
    predict_and_save([wav], out_dir, True, False, True, True, model)
    for ext in ("mid", "npz", "csv"):  # reference: tests/test_inference.py:79-102
        assert (out_dir / f"cfg1_basic_pitch.{ext}").is_file()
    with pytest.raises(IOError):
        predict_and_save([wav], out_dir, True, False, False, False, model)


def test_batch_position_and_chunking_invariance(model):
    """Size-independent property at scale: every window's result is independent of its position in the
    batch and of the internal chunking (300 windows = several chunks, one of them ragged)."""
    from basic_pitch_b200 import synth

    base = synth.window_batch(3, seed=5)
    x = np.tile(base, (100, 1))
    got = model.predict(x)
    for k in got:
        ref = got[k][:3]
        assert np.array_equal(got[k].reshape(100, 3, *ref.shape[1:]), np.broadcast_to(ref, (100,) + ref.shape)), k


def test_run_inference_equals_windowed_predict(model):
    """On-device windowing/unwrap == reference host windowing + per-window predict + unwrap, exactly."""
    from basic_pitch_b200 import synth
    from oracle import host_ref

    clips = [synth.random_notes_clip(10.0, seed=31), synth.tones_clip(2.0, seed=1), np.zeros(1, np.float32),
             synth.random_notes_clip(3.3, seed=33)[:36165]]
    # path 1 writes the unwrapped rows from the tap-sum kernels, paths 0 / 2 (partly) through separate copies
    for path in (1, 0, 2):
        try:
            model.set_path(path)
            outs = model.run_inference_arrays(clips)
            for clip, out in zip(clips, outs):
                raw = model.predict(host_ref.window_audio(clip))
                for k in raw:
                    np.testing.assert_array_equal(out[k], host_ref.unwrap(raw[k], len(clip)), err_msg=f"{k} (path {path})")
        finally:
            model.set_path(1)


def test_time_shift_equivariance_across_windows(model):
    """Size-independent property of the windowed pipeline: the overlap-and-drop scheme makes the unwrapped output
    (nearly) independent of where window boundaries fall.  A clip and the same clip delayed by exactly one window
    hop (36 164 samples = 142 frames of leading silence) must agree on the shifted frames to well below the decode
    thresholds away from the clip start."""
    from basic_pitch_b200 import synth

    clip = synth.random_notes_clip(8.0, seed=77)
    delayed = np.concatenate([np.zeros(36164, np.float32), clip])
    a, b = model.run_inference_arrays([clip, delayed])
    n = a["note"].shape[0] - 160
    for k in a:
        d = np.abs(a[k][150 : 150 + n - 150] - b[k][150 + 142 : 150 + 142 + n - 150])
        assert d.max() < 0.2 and d.mean() < 2e-3, (k, float(d.max()), float(d.mean()))


def test_transcribe_batch_equals_per_file(model):
    from basic_pitch_b200 import synth

    clips = [synth.random_notes_clip(6.0, seed=41), synth.dense_chords_clip(2.0, seed=3), synth.tones_clip(2.0, seed=2)]
    outs, res, frames = model.transcribe_arrays(clips)
    for i, c in enumerate(clips):
        o1, r1, f1 = model.transcribe_arrays([c])
        assert f1[0] == frames[i]
        for k in r1[0]:
            np.testing.assert_array_equal(r1[0][k], res[i][k], err_msg=k)
        for k in o1[0]:
            np.testing.assert_array_equal(o1[0][k], outs[i][k], err_msg=k)
    assert sum(len(r["start"]) for r in res) > 20


def test_transcribe_host_sub_batches_equal_device_path(model):
    """bp_transcribe_host splits a large batch into sub-batches on file boundaries (copies overlap the kernels) and runs
    partial internal chunks; its note events must equal those of one bp_transcribe_device call on the same audio, and the
    ragged file lengths exercise windows that cross sub-batch / chunk boundaries."""
    import torch

    from basic_pitch_b200 import engine, synth

    chunk = int(model._lib.bp_model_chunk_windows(model.handle))
    base = [synth.random_notes_clip(4.0 + 0.7 * (i % 5), seed=100 + i) for i in range(10)]
    clips = [base[i % len(base)] for i in range(160)]  # ~ 3 windows each -> several sub-batches of 1, 1, 2 chunks
    n_windows = sum(int(model._lib.bp_num_windows(len(c))) for c in clips)
    assert n_windows > 2 * chunk
    packed = engine.PackedAudio(clips, pinned=True)
    n_frames = sum(int(model._lib.bp_num_frames(len(c))) for c in clips)
    out_h = engine.NoteBuffers(len(clips), max(4096, 2 * n_frames), max(65536, 24 * n_frames))
    out_d = engine.NoteBuffers(len(clips), max(4096, 2 * n_frames), max(65536, 24 * n_frames))
    nh = engine.transcribe_packed_host(model, packed, out_h)
    d_audio = packed.to_device(model.device)
    nd = engine.transcribe_packed_device(model, d_audio, packed.offsets, out_d)
    torch.cuda.synchronize()
    assert nh == nd > 200
    for k in ("note_off", "frame_off"):
        np.testing.assert_array_equal(out_h.a[k][: len(clips) + 1], out_d.a[k][: len(clips) + 1], err_msg=k)
    for k in ("start", "end", "pitch", "amp"):
        np.testing.assert_array_equal(out_h.a[k][:nh], out_d.a[k][:nh], err_msg=k)
    nb = int(out_h.a["bend_off"][nh])
    np.testing.assert_array_equal(out_h.a["bend_off"][: nh + 1], out_d.a["bend_off"][: nh + 1])
    np.testing.assert_array_equal(out_h.a["bends"][:nb], out_d.a["bends"][:nb])
    # identical clips give identical events wherever they sit in the batch
    no = out_h.a["note_off"]
    for i in range(len(base), len(clips)):
        j = i % len(base)
        assert no[i + 1] - no[i] == no[j + 1] - no[j]
        np.testing.assert_array_equal(out_h.a["start"][no[i] : no[i + 1]], out_h.a["start"][no[j] : no[j + 1]])
        np.testing.assert_array_equal(out_h.a["amp"][no[i] : no[i + 1]], out_h.a["amp"][no[j] : no[j + 1]])


def test_get_infered_onsets_and_get_pitch_bends_entry_points(model):
    """The two sub-steps of the decode the reference also exposes as functions (note_creation.py:289-311, 182-219), through
    their own C-ABI entry points, bit-identical to the oracle restatements."""
    from basic_pitch_b200 import note_creation as nc
    from oracle import decode_ref

    rng = np.random.default_rng(5)
    T = 333  # not a multiple of the 32-frame tiles
    note = (rng.random((T, 88)) ** 3).astype(np.float32)
    onset = (rng.random((T, 88)) ** 4).astype(np.float32)
    got = nc.get_infered_onsets(onset, note, model=model)
    with np.errstate(all="ignore"):
        exp = decode_ref.infer_onsets(onset, note)
    assert got.dtype == np.float64 and got.shape == exp.shape
    np.testing.assert_array_equal(got, exp)
    # constant frames -> max(frame_diff) == 0 -> the reference's 0/0: an all-NaN matrix
    flat = np.full((40, 88), 0.25, np.float32)
    assert np.isnan(nc.get_infered_onsets(onset[:40], flat, model=model)).all()

    contour = rng.random((T, 264)).astype(np.float32)
    notes = []
    for _ in range(60):
        a = int(rng.integers(0, T - 2))
        b = int(rng.integers(a + 1, min(T, a + 90) + 1))
        notes.append((a, b, int(rng.integers(21, 109)), np.float32(rng.random())))
    notes += [(0, T, 21, np.float32(0.5)), (0, 1, 108, np.float32(0.5)), (T - 1, T, 60, np.float32(0.1))]
    got_b = nc.get_pitch_bends(contour, notes, model=model)
    exp_b = decode_ref.pitch_bends(contour, notes)
    assert len(got_b) == len(exp_b)
    for g, e in zip(got_b, exp_b):
        assert g[:3] == tuple(e[:3]) and g[3] == e[3]
        assert g[4] == [int(x) for x in e[4]]
    with pytest.raises(Exception):
        nc.get_pitch_bends(contour, [(5, 5, 60, 0.1)], model=model)  # empty note


def test_dense_polyphony_batch_bit_exact(model):
    """BASELINE configs[4]: 88-voice chords, several 10 s clips in one batch; decode (incl. pitch bends) bit-identical to
    the oracle decode on the same GPU posteriorgrams."""
    from basic_pitch_b200 import synth
    from oracle import decode_ref

    clips = [synth.dense_chords_clip(10.0, seed=7 + i) for i in range(3)]
    outs, res, frames = model.transcribe_arrays(clips)
    total = 0
    for i in range(len(clips)):
        with np.errstate(all="ignore"):
            wb, ev = decode_ref.model_output_to_note_events({k: np.array(v) for k, v in outs[i].items()}, 0.5, 0.3)
        exp = events_to_arrays(wb, ev)
        got_wb = [(int(a), int(b), int(p), amp, None) for a, b, p, amp in zip(res[i]["start"], res[i]["end"], res[i]["pitch"], res[i]["amp"])]
        from basic_pitch_b200 import note_creation as nc

        got = events_to_arrays(got_wb, nc.note_events_from_arrays(res[i], frames[i]))
        assert_events_equal(got, exp, ctx=f"chords clip {i}")
        total += len(ev)
    assert total > 300


def test_predict_batch_and_error_paths(model, tmp_path):
    import ctypes as C

    from basic_pitch_b200 import _lib, synth
    from basic_pitch_b200.inference import predict_batch

    clips = [synth.tones_clip(2.0, seed=3), synth.random_notes_clip(4.0, seed=5)]
    results = predict_batch(clips, model, multiple_pitch_bends=True)
    assert len(results) == 2
    for (out, midi, events), clip in zip(results, clips):
        assert out["note"].shape[0] == int(len(clip) / 36164 * 142)
        assert sum(len(i.notes) for i in midi.instruments) == len(events)
    # capacity negotiation: a deliberately tiny note buffer reports the needed size
    lib = _lib.load()
    post = model.run_inference_arrays([clips[1]])[0]
    notes, arrs = model._alloc_notes(1, 1, 1)
    p = model._params(0.5, 0.3, 11, 11, True, True, True, 0, 88)
    foff = np.array([0, post["note"].shape[0]], np.int64)
    with pytest.raises(_lib.BpError) as e:
        lib.bp_decode_host(model.handle, post["note"].ctypes.data, post["onset"].ctypes.data, post["contour"].ctypes.data,
                           foff.ctypes.data, 1, C.byref(p), C.byref(notes))
    assert e.value.code == _lib.BP_E_CAPACITY and "need" in str(e.value)
    # the reference never terminates for frame_thresh < 0 with melodia; this build refuses
    with pytest.raises(_lib.BpError) as e:
        model.decode_arrays([post["note"]], [post["onset"]], [post["contour"]], frame_thresh=-0.1)
    assert e.value.code == _lib.BP_E_INVALID
    # and the frequency limits zero the caller's arrays like the reference does
    from basic_pitch_b200 import note_creation as nc

    out = {k: np.array(v) for k, v in post.items()}
    nc.model_output_to_notes(out, 0.5, 0.3, min_freq=110.0, max_freq=880.0, model=model)
    lo, hi = nc.frequency_to_column_range(110.0, 880.0)
    assert not out["note"][:, :lo].any() and not out["onset"][:, hi:].any() and out["note"][:, lo:hi].any()


def test_two_models_with_different_weights_do_not_interfere(model, weights_np, tmp_path):
    """Weight-dependent constants live in __constant__ memory shared by all models of a process on one device; the library
    re-uploads them when the active model changes (the reference allows loading several model files side by side)."""
    from basic_pitch_b200 import synth, weights
    from basic_pitch_b200.inference import Model

    w2 = {k: v.copy() for k, v in weights_np.items()}
    w2["onset1_b"] = w2["onset1_b"] + 0.25
    w2["note2_w"] = w2["note2_w"] * 0.5
    w2["lowpass"] = w2["lowpass"][::-1].copy() * 0.9
    path = tmp_path / "other.bpw"
    path.write_bytes(weights.pack(w2))
    other = Model(path)
    x = synth.window_batch(3, seed=13)
    a0 = model.predict(x)
    b0 = other.predict(x)
    a1 = model.predict(x)
    b1 = other.predict(x)
    for k in a0:
        np.testing.assert_array_equal(a0[k], a1[k])
        np.testing.assert_array_equal(b0[k], b1[k])
    assert np.abs(a0["note"] - b0["note"]).max() > 1e-3 and np.abs(a0["onset"] - b0["onset"]).max() > 1e-3


@pytest.mark.gpu
def test_transcribe_files_host_equals_packed_entry_point(model):
    """bp_transcribe_files_host (one pointer per file, pageable memory, gathered and streamed per sub-batch by the library)
    returns bit-identical posteriorgrams and notes as bp_transcribe_host on the packed batch."""
    import ctypes as C

    from basic_pitch_b200 import _lib as L, synth

    lib = model._lib
    rng = np.random.default_rng(5)
    clips = [synth.tones_clip(float(rng.uniform(0.3, 7.0)), seed=40 + i) for i in range(23)] + [np.zeros(0, np.float32)]
    clips += [synth.tones_clip(31.0, seed=99)]
    n = len(clips)
    flat, offs = model._pack_audio(clips)
    frames = [int(lib.bp_num_frames(len(c))) for c in clips]
    total = sum(frames)
    p = model._params(0.5, 0.3, 11, 11, True, True, True, 0, 88)

    def run(files_api):
        note, onset = np.zeros((total, 88), np.float32), np.zeros((total, 88), np.float32)
        contour = np.zeros((total, 264), np.float32)
        foff = np.zeros(n + 1, np.int64)
        nt, arrs = model._alloc_notes(n, 4 * total, 64 * total)
        if files_api:
            ptrs = (C.c_void_p * n)(*[c.ctypes.data for c in clips])
            lens = np.array([len(c) for c in clips], np.int64)
            lib.bp_transcribe_files_host(model.handle, ptrs, lens.ctypes.data, n, C.byref(p), note.ctypes.data,
                                         onset.ctypes.data, contour.ctypes.data, foff.ctypes.data, C.byref(nt))
        else:
            lib.bp_transcribe_host(model.handle, flat.ctypes.data, offs.ctypes.data, n, C.byref(p), note.ctypes.data,
                                   onset.ctypes.data, contour.ctypes.data, foff.ctypes.data, C.byref(nt))
        k = int(arrs["note_off"][n])
        return note, onset, contour, foff, {a: arrs[a][:k].copy() for a in ("start", "end", "pitch", "amp")}, arrs["note_off"].copy()

    a, b = run(False), run(True)
    for x, y in zip(a[:4], b[:4]):
        np.testing.assert_array_equal(x, y)
    for key in a[4]:
        np.testing.assert_array_equal(a[4][key], b[4][key])
    np.testing.assert_array_equal(a[5], b[5])
    assert int(a[5][n]) > 50
    # degenerate batches through the Python mirror
    outs, res, frames = model.transcribe_arrays([])
    assert outs == [] and res == [] and frames == []
    outs, res, frames = model.transcribe_arrays([np.zeros(0, np.float32)])
    assert frames == [0] and outs[0]["note"].shape == (0, 88) and len(res[0]["start"]) == 0


@pytest.mark.gpu
def test_device_ingest_matches_host_loader(model, tmp_path):
    """csrc/ingest.cu (sample conversion + channel mean + polyphase resampler on the GPU, `load_audio_device`) against the
    host loader (`audio_io.load_audio`: NumPy + scipy.signal.resample_poly in float64) on WAV files of several formats."""
    from scipy.io import wavfile

    from basic_pitch_b200 import audio_io

    rng = np.random.default_rng(11)
    cases = [
        (44100, np.int16, 2, 70001), (48000, np.float32, 1, 50000), (16000, np.uint8, 1, 30011), (22050, np.int16, 2, 9999),
        (96000, np.int32, 2, 123457), (8000, np.int16, 1, 4000), (11025, np.float32, 3, 2048), (44100, np.int16, 1, 300),
    ]  # fmt: skip
    for i, (sr, dt, ch, n) in enumerate(cases):
        t = np.arange(n) / sr
        x = 0.4 * np.sin(2 * np.pi * 220.0 * t)[:, None] * np.linspace(1.0, 0.5, ch)[None, :] + 0.05 * rng.standard_normal((n, ch))
        if dt == np.float32:
            pcm = x.astype(np.float32)
        elif dt == np.uint8:
            pcm = np.clip(np.round(x * 127 + 128), 0, 255).astype(np.uint8)
        else:
            pcm = np.clip(np.round(x * (2.0 ** (8 * np.dtype(dt).itemsize - 1) - 1)), -(2.0 ** 31), 2.0 ** 31 - 1).astype(dt)
        if ch == 1:
            pcm = pcm[:, 0]
        path = tmp_path / f"c{i}.wav"
        wavfile.write(path, sr, pcm)
        ref, _ = audio_io.load_audio(path)
        got, sr_out = audio_io.load_audio_device(path, model)
        assert sr_out == 22050 and got.dtype == np.float32 and got.shape == ref.shape, (sr, dt, ch, got.shape, ref.shape)
        err = float(np.abs(got - ref).max()) if len(ref) else 0.0
        assert err < 3e-6, (sr, dt, ch, n, err)  # fp32 accumulation of ~400 taps vs float64


@pytest.mark.gpu
def test_device_ingest_vocadito_44k_vs_golden(model, golden_dir):
    """The reference's 44.1 kHz test clip through the device ingest and the model against the reference's golden
    posteriorgrams (reference: tests/test_inference.py:43-70; tolerance = the resampler residual, tests/golden/README.md)."""
    z = np.load(golden_dir / "vocadito10_pcm44k.npz")
    pcm, sr = z["pcm"], int(z["sample_rate"])
    lib = model._lib
    audio = np.empty(int(lib.bp_resampled_length(len(pcm), sr)), np.float32)
    lib.bp_load_pcm_host(model.handle, pcm.ctypes.data, 1, len(pcm), 1, sr, audio.ctypes.data)
    gold = load_vocadito(golden_dir)
    assert np.abs(audio - gold["audio22k"]).max() < 3e-6  # the host resampler of the fixture
    out = model.run_inference_arrays([audio])[0]
    for k in ("note", "onset", "contour"):
        assert out[k].shape == gold[f"gold_{k}"].shape
        assert float(np.abs(out[k] - gold[f"gold_{k}"]).max()) < GOLD_TOL, k


@pytest.mark.gpu
def test_streaming_mode_equals_whole_file(model):
    """Bounded-memory mode: run_inference_stream / predict_stream on a 70 s recording delivered in odd-sized blocks give
    the posteriorgrams of the whole-file call bit for bit, and the same note events."""
    from basic_pitch_b200 import synth
    from basic_pitch_b200.inference import predict_batch, predict_stream, run_inference_stream

    audio = synth.tones_clip(70.0, seed=21)
    whole = model.run_inference_arrays([audio])[0]
    blocks = [audio[p : p + 100003] for p in range(0, len(audio), 100003)]
    parts = list(run_inference_stream(blocks, model, windows_per_step=7))
    assert len(parts) > 5
    for k in ("note", "onset", "contour"):
        np.testing.assert_array_equal(np.concatenate([p[k] for p in parts]), whole[k])
    out, midi, events = predict_stream(blocks, model, windows_per_step=16)
    ref_out, _ref_midi, ref_events = predict_batch([audio], model, lazy=False)[0]
    np.testing.assert_array_equal(out["note"], ref_out["note"])
    assert len(events) > 20 and [e[:4] for e in events] == [e[:4] for e in ref_events]
    assert [list(e[4]) for e in events] == [list(e[4]) for e in ref_events]


@pytest.mark.gpu
def test_predict_and_save_batch_path(model, tmp_path):
    """predict_and_save over several files (batch path: GPU ingest, one device pass, bp_write_note_files) writes the same
    MIDI / CSV / NPZ files as the per-file path (`predict` + the Python writers)."""
    from scipy.io import wavfile

    from basic_pitch_b200 import inference as inf
    from basic_pitch_b200 import synth

    paths = []
    for i, (sr, secs) in enumerate(((22050, 3.0), (44100, 4.5), (22050, 0.7))):
        clip = synth.tones_clip(secs, seed=70 + i)
        if sr != 22050:
            clip = np.repeat(clip, 2)  # crude 44.1 kHz version: exercises the resampler on both paths
        p = tmp_path / f"clip{i}.wav"
        wavfile.write(p, sr, (clip * 20000).astype(np.int16))
        paths.append(p)
    out_b, out_s = tmp_path / "batch", tmp_path / "single"
    out_b.mkdir(), out_s.mkdir()
    inf.predict_and_save(paths, out_b, True, False, True, True, model)
    for p in paths:
        inf.predict_and_save([p], out_s, True, False, True, True, model)
    for p in paths:
        for ext in ("mid", "csv"):
            a = (out_b / f"{p.stem}_basic_pitch.{ext}").read_bytes()
            b = (out_s / f"{p.stem}_basic_pitch.{ext}").read_bytes()
            assert a == b and len(a) > 40, (p.name, ext)
        za = np.load(out_b / f"{p.stem}_basic_pitch.npz", allow_pickle=True)["basic_pitch_model_output"].item()
        zb = np.load(out_s / f"{p.stem}_basic_pitch.npz", allow_pickle=True)["basic_pitch_model_output"].item()
        for k in ("note", "onset", "contour"):
            np.testing.assert_array_equal(za[k], zb[k])

