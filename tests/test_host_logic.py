"""CPU: host-side logic of the drop-in (no GPU): weights, constants, time mapping, MIDI assembly, audio I/O."""
import numpy as np
import pytest

from oracle import decode_ref
from tests.golden_util import load_vocadito


def test_weight_blob_roundtrip_and_dsp_constants(weights_np):
    from basic_pitch_b200 import weights

    blob = weights.pack(weights_np)
    again = weights.unpack(blob)
    for k, v in weights_np.items():
        np.testing.assert_array_equal(again[k], v)
    dsp = weights.dsp_constants()
    for k in ("cqt_real", "cqt_imag", "lowpass", "cqt_scale"):
        np.testing.assert_array_equal(dsp[k], weights_np[k], err_msg=k)  # SURVEY Appendix A.1: bit-identical
    # fingerprints, SURVEY Appendix A.4
    assert abs(float(weights_np["onset1_w"].astype("f8").sum()) - 5.7735) < 1e-4
    assert abs(float(weights_np["contour1_w"].astype("f8").sum()) - 2.75278) < 1e-4
    assert abs(float(weights_np["note1_b"].astype("f8").sum()) - 7.64196) < 1e-4


def test_bad_model_file_raises_valueerror(tmp_path):
    from basic_pitch_b200.inference import Model

    p = tmp_path / "junk.onnx"
    p.write_bytes(b"\x08\x01\x12\x04junk")
    with pytest.raises(ValueError):
        Model(p)


def test_constants_match_reference_values():
    from basic_pitch_b200 import constants as c

    assert (c.FFT_HOP, c.AUDIO_SAMPLE_RATE, c.ANNOTATIONS_FPS, c.ANNOT_N_FRAMES, c.AUDIO_N_SAMPLES) == (256, 22050, 86, 172, 43844)
    assert (c.N_FREQ_BINS_NOTES, c.N_FREQ_BINS_CONTOURS, c.HOP_SIZE, c.FRAMES_PER_HOP) == (88, 264, 36164, 142)


def test_frames_to_time_matches_oracle():
    from basic_pitch_b200.note_creation import model_frames_to_time

    for n in (0, 1, 171, 172, 173, 787, 15584):
        np.testing.assert_array_equal(model_frames_to_time(n), decode_ref.frames_to_time(n))


@pytest.mark.parametrize("mn,mx", [(None, None), (110.0, 880.0), (20.0, None), (None, 20000.0), (5000.0, 100.0), (27.5, 4186.0)])
def test_frequency_range_follows_numpy_slicing(mn, mx):
    from basic_pitch_b200.note_creation import constrain_frequency, frequency_to_column_range

    a = np.ones((3, 88), np.float32)
    b = np.ones((3, 88), np.float32)
    decode_ref.constrain_frequency(a, b, mx, mn)
    lo, hi = frequency_to_column_range(mn, mx)
    keep = np.zeros(88, bool)
    keep[lo:hi] = True
    np.testing.assert_array_equal(a[0] != 0, keep)
    c = np.ones((3, 88), np.float32)
    d = np.ones((3, 88), np.float32)
    constrain_frequency(c, d, mx, mn)
    np.testing.assert_array_equal(c, a)
    np.testing.assert_array_equal(d, b)


def test_drop_overlapping_pitch_bends_reference_case():
    """The hand-made case of reference: tests/test_note_creation.py:21-50."""
    from basic_pitch_b200.note_creation import drop_overlapping_pitch_bends

    ev = [
        (0.0, 0.1, 1, 1.0, [0, 1, 2]),
        (2.0, 2.1, 1, 1.0, [0, 1, 2]),  # overlaps the next
        (2.0, 2.1, 1, 1.0, [0, 1, 2]),
        (3.0, 3.2, 1, 1.0, [0, 1, 2]),  # overlaps 3.1-3.3
        (3.1, 3.3, 1, 1.0, [0, 1, 2]),
        (5.0, 5.1, 1, 1.0, [0, 1, 2]),
        (5.1, 5.2, 1, 1.0, [0, 1, 2]),  # touching is not overlapping
    ]
    out = drop_overlapping_pitch_bends(ev)
    got = [e[4] is None for e in out]
    assert got == [False, True, True, True, True, False, False]
    assert out == decode_ref.drop_overlapping_pitch_bends(ev)


def test_note_events_to_midi_and_smf_writer(tmp_path):
    from basic_pitch_b200 import note_creation as nc

    events = [
        (0.5, 1.0, np.int64(60), np.float32(0.5), [0, 1, -1, 3]),
        (2.0, 2.5, np.int64(64), np.float32(0.996), None),
        (0.7, 0.9, np.int64(67), np.float32(0.1), [5, 5]),  # overlaps the first -> both lose bends
    ]
    mid = nc.note_events_to_midi(events, multiple_pitch_bends=False, midi_tempo=120)
    (inst,) = mid.instruments
    assert inst.program == 4
    assert sorted((n.pitch, n.velocity) for n in inst.notes) == [(60, 64), (64, 126), (67, 13)]
    assert inst.pitch_bends == []
    mid2 = nc.note_events_to_midi(events, multiple_pitch_bends=True)
    assert len(mid2.instruments) == 3
    bends = [b.pitch for i in mid2.instruments for b in i.pitch_bends]
    assert bends == [0, 1365, -1365, 4096, 6827, 6827]
    path = tmp_path / "x.mid"
    mid2.write(str(path))
    raw = path.read_bytes()
    assert raw[:4] == b"MThd" and raw.count(b"MTrk") == 4


def test_audio_io_wav_and_resample(tmp_path):
    from scipy.io import wavfile

    from basic_pitch_b200.audio_io import load_audio

    sr = 22050
    t = np.arange(sr) / sr
    x = (0.5 * np.sin(2 * np.pi * 440 * t)).astype(np.float32)
    p = tmp_path / "a.wav"
    wavfile.write(p, sr, (x * 32767).astype(np.int16))
    y, r = load_audio(p)
    assert r == 22050 and y.dtype == np.float32 and y.shape == x.shape
    assert np.abs(y - x).max() < 1e-4
    st = np.stack([x, -x * 0.5], axis=1)
    p2 = tmp_path / "b.wav"
    wavfile.write(p2, 44100, np.repeat(st, 2, axis=0))
    y2, _ = load_audio(p2)
    assert abs(len(y2) - len(x)) <= 1
    assert np.abs(y2[100:-100] - 0.25 * x[100 : len(y2) - 100]).max() < 2e-2


def test_window_and_unwrap_helpers_match_oracle():
    from basic_pitch_b200 import inference as inf
    from oracle import host_ref

    x = np.random.default_rng(0).standard_normal(100000).astype(np.float32)
    xw = np.concatenate([np.zeros(3840, np.float32), x])
    wins = np.concatenate([w[None, :, 0] for w, _ in inf.window_audio_file(xw, 36164)])
    np.testing.assert_array_equal(wins, host_ref.window_audio(x))
    out = np.random.default_rng(1).random((wins.shape[0], 172, 5)).astype(np.float32)
    np.testing.assert_array_equal(inf.unwrap_output(out, len(x), 30, 36164), host_ref.unwrap(out, len(x)))


def test_numpy_pairwise_sum_model():
    """The summation order implemented in csrc/decode.cu::np_pairwise_sum, restated in Python, must equal
    np.mean on strided float32 columns (this is what makes GPU amplitudes bit-identical)."""

    def pw(a):
        n = len(a)
        f = np.float32
        if n < 8:
            r = f(0)
            for v in a:
                r = f(r + v)
            return r
        if n <= 128:
            r = [f(v) for v in a[:8]]
            i = 8
            while i < n - (n % 8):
                for j in range(8):
                    r[j] = f(r[j] + a[i + j])
                i += 8
            res = f(f(f(r[0] + r[1]) + f(r[2] + r[3])) + f(f(r[4] + r[5]) + f(r[6] + r[7])))
            while i < n:
                res = f(res + a[i])
                i += 1
            return res
        n2 = n // 2
        n2 -= n2 % 8
        return f(pw(a[:n2]) + pw(a[n2:]))

    rng = np.random.default_rng(5)
    m = rng.random((3100, 88)).astype(np.float32)
    for n in (1, 2, 7, 8, 9, 15, 16, 17, 100, 127, 128, 129, 130, 255, 256, 257, 1000, 1023, 2999):
        col = m[5 : 5 + n, 17]
        assert np.float32(pw(col) / np.float32(n)) == np.mean(col), n


def test_decode_substep_functions_reject_unsupported_arguments():
    """get_pitch_bends / get_infered_onsets exist with the reference's signatures (note_creation.py:182, 289); the device
    kernels implement the reference defaults only, other values are refused before any GPU work."""
    from basic_pitch_b200 import note_creation as nc

    with pytest.raises(NotImplementedError):
        nc.get_pitch_bends(np.zeros((4, 264), np.float32), [(0, 2, 60, 0.5)], n_bins_tolerance=10)
    with pytest.raises(NotImplementedError):
        nc.get_infered_onsets(np.zeros((4, 88), np.float32), np.zeros((4, 88), np.float32), n_diff=3)
    assert nc.SONIFY_FS == 3000


def test_sonification_helpers(tmp_path):
    """sonify_midi / sonify_salience (reference: note_creation.py:119-165): same signatures, files and return values; the
    synthesis itself restates pretty_midi / mir_eval behaviour (sum of sinusoids, peak-normalised)."""
    from scipy.io import wavfile

    from basic_pitch_b200 import note_creation as nc

    ev = [(0.1, 0.6, 69, np.float32(0.8), [0, 1, 2, 1, 0]), (0.3, 1.0, 76, np.float32(0.5), None)]
    for midi in (nc.note_events_to_midi(ev), nc.LazyPrettyMIDI(ev)):
        path = tmp_path / "m.wav"
        nc.sonify_midi(midi, path, 8000)
        sr, y = wavfile.read(path)
        assert sr == 8000 and len(y) == int(8000 * (1.0 + 1)) and abs(np.abs(y).max() - 1.0) < 1e-9
        seg = y[int(0.12 * sr) : int(0.28 * sr)]  # only the A4 sounds here
        f = np.fft.rfftfreq(len(seg), 1 / sr)
        assert abs(f[np.abs(np.fft.rfft(seg * np.hanning(len(seg)))).argmax()] - 440.0) < 12.0
    gram = np.zeros((264, 100))
    gram[60, 10:50] = 0.9
    gram[120, 30:80] = 0.5
    gram[200, :] = 0.1  # below thresh: zeroed in place
    y, fs = nc.sonify_salience(gram, 3, str(tmp_path / "s.wav"))
    assert fs == 3000 and gram[200].max() == 0 and abs(np.abs(y).max() - 1.0) < 1e-9
    f = np.fft.rfftfreq(len(y), 1 / fs)
    assert abs(f[np.abs(np.fft.rfft(y)).argmax()] - 27.5 * 2 ** (60 / 36)) < 1.0
    sr, y44 = wavfile.read(tmp_path / "s.wav")
    assert sr == 44100 and abs(len(y44) - len(y) * 44100 / 3000) <= 1


def test_file_output_helpers_match_reference_behaviour(tmp_path):
    """save_note_events / build_output_path / verify_* (reference: inference.py:349-428).  Expected strings were produced by
    the unmodified reference functions (oracle/ref_shims) on the same inputs."""
    import pathlib

    from basic_pitch_b200 import inference as inf

    ev = [(np.float64(0.5), np.float64(1.25), np.int64(60), np.float32(0.73), [np.int64(1), np.int64(-2), np.int64(0)]),
          (np.float64(0.011609977324263039), np.float64(0.13), np.int64(21), np.float32(0.004), None),
          (np.float64(2.0), np.float64(2.5), np.int64(108), np.float32(1.0), [])]
    p = tmp_path / "x.csv"
    inf.save_note_events(ev, p)
    assert p.read_text() == ("start_time_s,end_time_s,pitch_midi,velocity,pitch_bend\n0.5,1.25,60,93,1,-2,0\n"
                             "0.011609977324263039,0.13,21,1\n2.0,2.5,108,127\n")
    assert [(e.name, e.value) for e in inf.OutputExtensions] == [
        ("MIDI", "mid"), ("MODEL_OUTPUT_NPZ", "npz"), ("MIDI_SONIFICATION", "wav"), ("NOTE_EVENTS", "csv")]
    assert inf.build_output_path("/a/b/song.flac", str(tmp_path), inf.OutputExtensions.MIDI) == tmp_path / "song_basic_pitch.mid"
    assert inf.build_output_path("song.name.wav", tmp_path, inf.OutputExtensions.NOTE_EVENTS) == tmp_path / "song.name_basic_pitch.csv"
    (tmp_path / "song_basic_pitch.mid").write_text("x")
    with pytest.raises(IOError):
        inf.build_output_path("/x/song.wav", tmp_path, inf.OutputExtensions.MIDI)
    for fn, arg in ((inf.verify_input_path, tmp_path / "nope.wav"), (inf.verify_input_path, tmp_path),
                    (inf.verify_output_dir, tmp_path / "nodir"), (inf.verify_output_dir, p)):
        with pytest.raises(ValueError):
            fn(arg)
    inf.verify_input_path(p)
    inf.verify_output_dir(pathlib.Path(tmp_path))


def test_window_audio_file_and_get_audio_input_like_the_reference_tests(golden_dir, tmp_path):
    """Mirrors reference tests/test_inference.py:164-194 (`test_window_audio_file`, `test_get_audio_input`) on the same
    recording (its 22 050 Hz rendition from the golden fixture; a float32 WAV round-trips exactly)."""
    from scipy.io import wavfile

    from basic_pitch_b200 import inference as inf
    from basic_pitch_b200.constants import AUDIO_N_SAMPLES, AUDIO_SAMPLE_RATE, FFT_HOP

    audio = load_vocadito(golden_dir)["audio22k"]
    windows, times = zip(*inf.window_audio_file(audio, AUDIO_N_SAMPLES - 30 * FFT_HOP))
    assert len(windows) == 6 and len(times) == 6
    assert all(t["start"] <= t["end"] for t in times)
    np.testing.assert_equal(audio[:AUDIO_N_SAMPLES], np.squeeze(windows[0]))

    wav = tmp_path / "vocadito_10_22k.wav"
    wavfile.write(wav, AUDIO_SAMPLE_RATE, audio)  # float32 WAV
    overlap_len = 30 * FFT_HOP
    padded = np.concatenate([np.zeros((overlap_len // 2,), dtype=np.float32), audio])
    got, got_times, orig = [], [], None
    for w, t, original_length in inf.get_audio_input(wav, overlap_len, AUDIO_N_SAMPLES - overlap_len):
        got.append(w)
        got_times.append(t)
        orig = original_length
    got = np.array(got)
    assert len(got) == 6 and len(got_times) == 6
    assert all(t["start"] <= t["end"] for t in got_times)
    np.testing.assert_equal(padded[:AUDIO_N_SAMPLES], np.squeeze(got[0]))
    assert orig == 200607
    with pytest.raises(AssertionError):
        next(inf.get_audio_input(wav, 3, AUDIO_N_SAMPLES - 3))  # odd overlap, like the reference (inference.py:237)


def test_ingest_filter_and_length_match_scipy():
    """The device resampler (csrc/ingest.cu) designs its Kaiser low-pass itself: same taps as audio_io._resample_filter
    (scipy.signal.kaiserord + firwin) and the output length of scipy.signal.resample_poly."""
    import scipy.signal

    from basic_pitch_b200 import _lib, audio_io

    lib = _lib.load()
    for up, down in ((1, 2), (147, 320), (441, 160), (147, 640)):
        ref = audio_io._resample_filter(up, down)
        n = int(lib.bp_debug_resample_filter(up, down, None, 0))
        assert n == len(ref)
        h = np.zeros(n)
        lib.bp_debug_resample_filter(up, down, h.ctypes.data, n)
        assert np.abs(h - ref).max() < 1e-14
    for sr, n in ((44100, 401214), (48000, 12345), (16000, 777), (8000, 1), (22050, 99), (96000, 100001)):
        g = np.gcd(22050, sr)
        ref_len = len(scipy.signal.resample_poly(np.zeros(n), 22050 // g, sr // g)) if sr != 22050 else n
        assert int(lib.bp_resampled_length(n, sr)) == ref_len


@pytest.mark.parametrize("multi,tempo", [(False, 120.0), (True, 120.0), (False, 97.5)])
def test_batched_writers_are_byte_identical_to_the_python_path(tmp_path, multi, tempo):
    """csrc/writers.cu (`bp_write_note_files` through note_creation.write_note_files): the MIDI and CSV files of a batch,
    written by host threads straight from the note arrays, against note_events_to_midi(...).write() /
    save_note_events per file (reference: note_creation.py:222-286, inference.py:409-428) — ties, overlapping notes
    (dropped pitch bends), empty files, one- and zero-length bend lists included."""
    from basic_pitch_b200 import inference as inf
    from basic_pitch_b200 import note_creation as nc

    rng = np.random.default_rng(1)
    n_files = 9
    per = rng.integers(0, 60, n_files)
    per[3] = 0
    noff = np.zeros(n_files + 1, np.int32)
    noff[1:] = np.cumsum(per)
    n = int(noff[-1])
    start = rng.integers(0, 600, n).astype(np.int32)
    end = start + rng.integers(11, 60, n).astype(np.int32)
    start[5:9] = start[5]
    end[5:7] = end[5]
    bl = end - start
    bl[10], bl[11] = 1, 0
    boff = np.zeros(n + 1, np.int32)
    boff[1:] = np.cumsum(bl)
    arrs = dict(note_off=noff, start=start, end=end, pitch=rng.integers(21, 108, n).astype(np.int32),
                amp=rng.random(n).astype(np.float32), bend_off=boff, bends=rng.integers(-40, 40, boff[-1]).astype(np.int32))
    arrs["pitch"][5:7] = 60
    arrs["amp"][5:7] = 0.5
    lazy = nc.note_events_batch(arrs, n_files)
    eager = nc.note_events_batch(arrs, n_files, lazy=False)
    for tag, events in (("lazy", lazy), ("eager", eager)):
        mp = [tmp_path / f"{tag}{i}.mid" for i in range(n_files)]
        cp = [tmp_path / f"{tag}{i}.csv" for i in range(n_files)]
        mp[2] = None  # skipped
        nc.write_note_files(events, mp, cp, multiple_pitch_bends=multi, midi_tempo=tempo, n_threads=3)
        for i in range(n_files):
            nc.note_events_to_midi(eager[i], multi, tempo).write(str(tmp_path / "ref.mid"))
            inf.save_note_events(eager[i], tmp_path / "ref.csv")
            if mp[i] is not None:
                assert mp[i].read_bytes() == (tmp_path / "ref.mid").read_bytes(), (tag, i)
            else:
                assert not (tmp_path / f"{tag}{i}.mid").exists()
            assert cp[i].read_bytes() == (tmp_path / "ref.csv").read_bytes(), (tag, i)


def test_note_event_list_behaves_like_the_list():
    from basic_pitch_b200 import note_creation as nc

    noff = np.array([0, 3, 3, 5], np.int32)
    arrs = dict(note_off=noff, start=np.array([1, 5, 9, 2, 4], np.int32), end=np.array([20, 30, 25, 14, 40], np.int32),
                pitch=np.array([60, 62, 64, 40, 41], np.int32), amp=np.array([.1, .2, .3, .4, .5], np.float32),
                bend_off=np.array([0, 2, 2, 5, 6, 6], np.int32), bends=np.array([1, -1, 3, 0, 2, 7], np.int32))
    lazy, eager = nc.note_events_batch(arrs, 3), nc.note_events_batch(arrs, 3, lazy=False)
    assert [len(x) for x in lazy] == [3, 0, 2]
    for a, b in zip(lazy, eager):
        assert a == b and list(a) == b and a[:] == b and sorted(a) == sorted(b)
        if len(b):
            assert a[-1] == b[-1] and a[0][4] == b[0][4]
    assert lazy[0][0][4] == [1, -1] and lazy[0][1][4] == [] and lazy[2][1][4] == []
    with pytest.raises(IndexError):
        lazy[1][0]
    m = nc.LazyPrettyMIDI(lazy[0])
    assert len(m.instruments) == 1 and len(m.instruments[0].notes) == 3


def test_streaming_windowing_equals_whole_file_windowing():
    """run_inference_stream (bounded-memory mode, reference: README.md:196-198): block-wise windowing, the two-window
    hold-back and the final trim reproduce window_audio_file + unwrap_output (inference.py:194-279) for every length /
    block pattern — checked with a stand-in model on the CPU (the GPU test runs the real one)."""
    from basic_pitch_b200 import inference as inf

    class FakeModel(inf.Model):
        def __init__(self):
            pass

        def __del__(self):
            pass

        def predict(self, x):
            x = np.asarray(x)
            fr = np.stack([x[:, t * 255 : t * 255 + 256].mean(axis=1) for t in range(172)], axis=1).astype(np.float32)
            return {"note": np.repeat(fr[:, :, None], 88, 2), "onset": np.repeat(2 * fr[:, :, None], 88, 2),
                    "contour": np.repeat(3 * fr[:, :, None], 264, 2)}

    m = FakeModel()
    rng = np.random.default_rng(0)
    hop = 43844 - 30 * 256
    for n in (0, 1, 3840, hop - 3840, hop - 3839, hop, hop + 1, 2 * hop - 100, 5 * hop + 17, 7 * hop):
        audio = rng.standard_normal(n).astype(np.float32)
        padded = np.concatenate([np.zeros(3840, np.float32), audio])
        wins = [w[:, 0] for w, _ in inf.window_audio_file(padded, hop)]
        ref = {k: inf.unwrap_output(v, n, 30, hop) for k, v in m.predict(np.stack(wins)).items()} if wins else None
        for block in (max(n, 1), 50000, 9973):
            blocks = [audio[p : p + block] for p in range(0, n, block)]
            parts = list(inf.run_inference_stream(blocks, m, windows_per_step=3))
            for k, width in (("note", 88), ("onset", 88), ("contour", 264)):
                got = np.concatenate([q[k] for q in parts]) if parts else np.zeros((0, width), np.float32)
                want = ref[k] if ref is not None else np.zeros((0, width), np.float32)
                assert got.shape == want.shape and np.array_equal(got, want), (n, block, k)


def test_batched_writer_reports_unwritable_paths(tmp_path):
    """bp_write_note_files: a path that cannot be opened is an error (BpError), files before it are still written."""
    from basic_pitch_b200 import _lib
    from basic_pitch_b200 import note_creation as nc

    ev = [[(0.1, 0.5, 60, np.float32(0.5), [0, 1])], [(0.2, 0.9, 62, np.float32(0.7), None)]]
    good, bad = tmp_path / "a.mid", tmp_path / "no_such_dir" / "b.mid"
    with pytest.raises(_lib.BpError):
        nc.write_note_files(ev, [good, bad], None, n_threads=1)
    assert good.exists() and not bad.exists()
    nc.write_note_files([], [], [])  # an empty batch is fine
