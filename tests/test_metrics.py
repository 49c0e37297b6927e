"""Speech-quality metrics (deepfilternet_b200.metrics, dfb_metrics) against tests/golden/metrics.npz, the values of the
reference's own df.stoi.stoi, df.sepm.SNRseg / llr / wss and si_sdr_speechmetrics (oracle/gen_golden_metrics.py).

Tolerances:
  STOI    1e-4 absolute: the reference's known-answer tolerance (tests/test_df.py:18-19 of the reference).
  SI-SDR / segmental SNR   1e-3 dB.
  LLR     1e-4 relative (+ 1e-6 absolute for values at 0): sepm.lpcoeff rounds the autocorrelation and the LPC
          coefficients to float32 and llr forms the quadratic forms A' R A in float32 BLAS; the device forms them in
          fp64 from the same float32-rounded values, so the reference's own rounding of those forms is the difference
          (2e-5 relative on the DeepFilterNet3 pair, below 5e-6 on the others).
  WSS     1e-4 relative (+ 1e-6 absolute): the 1024-point FFT is fp32 on the device, float64 in scipy (2e-7 relative).
"""
import os

import numpy as np
import pytest
import torch

import ref_harness as rh

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ASSETS = os.path.join(GOLD, "assets")
COLS = ("stoi", "sisdr", "ssnr", "llr", "wss")


def fixture():
    return np.load(os.path.join(GOLD, "metrics.npz"))


def pair_inputs(g, i):
    """(clean, degraded, sr) of fixture pair i as float32 numpy arrays (48 kHz pairs; asset16 is resampled here)."""
    name = str(g["names"][i])
    if f"p{i}_clean" in g:
        return g[f"p{i}_clean"].astype(np.float32) / 32768, g[f"p{i}_deg"].astype(np.float32) / 32768, int(g["rates"][i])
    if name.startswith("asset"):
        c = rh.read_wav(os.path.join(ASSETS, "clean_freesound_33711.wav"))[0]
        n = rh.read_wav(os.path.join(ASSETS, "noisy_snr0.wav"))[0]
        if name == "asset16":
            from deepfilternet_b200.io import resample
            c = resample(torch.from_numpy(c)[None], 48000, 16000)[0].numpy()
            n = resample(torch.from_numpy(n)[None], 48000, 16000)[0].numpy()
        return c, n, int(g["rates"][i])
    ch = int(name.split("_")[1])
    d3 = np.load(os.path.join(GOLD, "dfnet_DeepFilterNet3.npz"))
    return d3["audio"][ch], d3["enhanced"][ch], 48000


def assert_matches(got, ref, name):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    tol = {"stoi": (1e-4, 0.0), "sisdr": (1e-3, 0.0), "ssnr": (1e-3, 0.0), "llr": (1e-6, 1e-4), "wss": (1e-6, 1e-4)}
    for j, m in enumerate(COLS):
        a, r = got[j], ref[j]
        if np.isnan(r):
            assert np.isnan(a), (name, m, a, r)
            continue
        atol, rtol = tol[m]
        assert abs(a - r) <= atol + rtol * abs(r), (name, m, a, r, abs(a - r))


# ---------------------------------------------------------------------------------------------- CPU ----
def test_fixture_layout_and_si_sdr_restatement():
    """The fixture is small and self-consistent: its SI-SDR values agree with oracle/ref_harness.si_sdr (the
    restatement the other tests use) on every stored pair, and the too-short pair has no STOI."""
    assert os.path.getsize(os.path.join(GOLD, "metrics.npz")) < 1 << 20
    g = fixture()
    names = [str(n) for n in g["names"]]
    assert tuple(str(m) for m in g["metrics"]) == COLS and g["values"].shape == (len(names), 5)
    stored = [i for i in range(len(names)) if f"p{i}_clean" in g]
    assert len(stored) >= 9
    for i in stored:
        c, d, _ = pair_inputs(g, i)
        assert abs(rh.si_sdr(c, d) - g["values"][i, 1]) < 1e-4, names[i]
    assert np.isnan(g["values"][names.index("short"), 0])
    assert len({len(pair_inputs(g, names.index(f"ragged{k}"))[0]) for k in range(4)}) == 4
    ident = g["values"][names.index("identical")]
    assert ident[0] == pytest.approx(1.0, abs=1e-6) and ident[2] == 35.0 and ident[4] == 0.0


def test_arguments_are_checked_before_any_device_call(monkeypatch):
    from deepfilternet_b200 import _lib, metrics

    def no_device():
        raise AssertionError("the library was reached")

    monkeypatch.setattr(_lib, "lib", no_device)
    x = torch.zeros(2, 1000)
    with pytest.raises(ValueError, match="lengths"):
        metrics.evaluate(x, x, 16000, lengths=[1000, 1001])
    with pytest.raises(ValueError, match="lengths"):
        metrics.evaluate(x, x, 16000, lengths=[0, 10])
    with pytest.raises(ValueError, match="lengths"):
        metrics.evaluate(x, x, 16000, lengths=[10])
    with pytest.raises(ValueError, match="sample rate"):
        metrics.evaluate(x, x, 12345)
    with pytest.raises(ValueError, match="unknown metrics"):
        metrics.evaluate(x, x, 16000, metrics=("pesq",))
    with pytest.raises(ValueError, match="shapes differ"):
        metrics.evaluate(x, torch.zeros(2, 999), 16000)
    with pytest.raises(ValueError, match="16 kHz"):
        metrics.wss(x[0], x[0], 48000)
    with pytest.raises(AssertionError):
        metrics.stoi(x[0], x[0], 16000)


def test_c_abi_rejects_bad_arguments():
    """dfb_metrics_host validates on the host, before it selects a device (DFB_ERR_INVALID, -1)."""
    import ctypes as C

    from deepfilternet_b200 import _lib
    L = _lib.lib()
    x = np.zeros((2, 100), np.float32)
    out = np.zeros((2, 5), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    for lens, sr, which in (([100, 101], 16000, 31), ([0, 10], 16000, 31), ([10, 10], 11025, 31), ([10, 10], 16000, 0),
                            ([10, 10], 16000, 32)):
        ln = np.array(lens, np.int64)
        assert L.dfb_metrics_host(0, p(x), p(x), p(ln), 2, 100, sr, which, p(out)) == _lib.DFB_ERR_INVALID
        assert L.dfb_last_error()


# ---------------------------------------------------------------------------------------------- GPU ----
@pytest.mark.gpu
def test_every_metric_against_the_reference():
    from deepfilternet_b200 import metrics
    g = fixture()
    for i, name in enumerate(str(n) for n in g["names"]):
        c, d, sr = pair_inputs(g, i)
        got = metrics.evaluate(torch.from_numpy(c), torch.from_numpy(d), sr)
        assert_matches([float(got[m][0]) for m in COLS], g["values"][i], name)


@pytest.mark.gpu
def test_single_pair_functions():
    from deepfilternet_b200 import metrics
    g = fixture()
    names = [str(n) for n in g["names"]]
    i = names.index("ragged2")
    c, d, _ = pair_inputs(g, i)
    ref = g["values"][i]
    got = [float(metrics.stoi(torch.from_numpy(c)[None], torch.from_numpy(d)[None], 16000)[0]), metrics.si_sdr(c, d),
           metrics.ssnr(c, d, 16000), metrics.llr(c, d, 16000), metrics.wss(c, d, 16000)]
    assert_matches(got, ref, "ragged2")
    s = metrics.stoi(torch.from_numpy(c)[None].cuda(), torch.from_numpy(d)[None].cuda(), 16000)
    assert s.device.type == "cuda" and s.shape == (1,)


def _synthetic_batch(g, rng):
    names = [str(n) for n in g["names"]]
    idx = [i for i in range(len(names)) if f"p{i}_clean" in g]
    pairs = [pair_inputs(g, i)[:2] for i in idx]
    T = max(len(c) for c, _ in pairs)
    # padding holds noise: nothing past lengths[b] may reach a result
    x = rng.standard_normal((len(pairs), T)).astype(np.float32)
    y = rng.standard_normal((len(pairs), T)).astype(np.float32)
    for b, (c, d) in enumerate(pairs):
        x[b, :len(c)], y[b, :len(d)] = c, d
    return idx, pairs, x, y, [len(c) for c, _ in pairs]


@pytest.mark.gpu
def test_ragged_batch_equals_each_pair_alone_and_matches_reference():
    from deepfilternet_b200 import metrics
    g = fixture()
    idx, pairs, x, y, lens = _synthetic_batch(g, np.random.default_rng(0))
    batch = metrics.evaluate(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), 16000, lengths=lens)
    assert all(v.device.type == "cuda" and v.shape == (len(idx),) for v in batch.values())
    got = np.stack([batch[m].cpu().numpy() for m in COLS], 1)
    for b, (c, d) in enumerate(pairs):
        alone = metrics.evaluate(torch.from_numpy(c), torch.from_numpy(d), 16000)
        np.testing.assert_array_equal(got[b], np.array([float(alone[m][0]) for m in COLS], np.float32))
        assert_matches(got[b], g["values"][idx[b]], str(g["names"][idx[b]]))
    # the list form pads and takes the lengths itself
    as_list = metrics.evaluate([torch.from_numpy(c) for c, _ in pairs], [torch.from_numpy(d) for _, d in pairs], 16000)
    np.testing.assert_array_equal(np.stack([as_list[m].numpy() for m in COLS], 1), got)
    # a subset of the metrics gives the same values
    sub = metrics.evaluate(torch.from_numpy(x), torch.from_numpy(y), 16000, lengths=lens, metrics=("wss", "stoi"))
    assert list(sub) == ["wss", "stoi"]
    np.testing.assert_array_equal(sub["wss"].numpy(), got[:, 4])
    np.testing.assert_array_equal(sub["stoi"].numpy(), got[:, 0])


@pytest.mark.gpu
def test_permuting_the_batch_permutes_the_results():
    from deepfilternet_b200 import metrics
    g = fixture()
    _, _, x, y, lens = _synthetic_batch(g, np.random.default_rng(1))
    perm = np.random.default_rng(2).permutation(len(lens))
    a = metrics.evaluate(torch.from_numpy(x), torch.from_numpy(y), 16000, lengths=lens)
    b = metrics.evaluate(torch.from_numpy(x[perm]), torch.from_numpy(y[perm]), 16000, lengths=np.array(lens)[perm])
    for m in COLS:
        np.testing.assert_array_equal(b[m].numpy(), a[m].numpy()[perm])


@pytest.mark.gpu
def test_too_short_for_stoi_is_nan():
    from deepfilternet_b200 import metrics
    g = fixture()
    c, d, _ = pair_inputs(g, [str(n) for n in g["names"]].index("short"))
    r = metrics.evaluate(torch.from_numpy(c), torch.from_numpy(d), 16000)
    assert np.isnan(float(r["stoi"][0]))
    assert all(np.isfinite(float(r[m][0])) for m in COLS[1:])
    # below 600 samples at 16 kHz no 30 ms frame is scored: the sepm measures are NaN too
    r = metrics.evaluate(torch.from_numpy(c[:599]), torch.from_numpy(d[:599]), 16000)
    assert all(np.isnan(float(r[m][0])) for m in ("stoi", "ssnr", "llr", "wss")) and np.isfinite(float(r["sisdr"][0]))


@pytest.mark.gpu
def test_enhance_output_scored_on_the_device(model_dir):
    """enhance() on the DeepFilterNet3 fixture input (seeded random weights), scored on the device against its input,
    gives the reference's values for the reference's enhanced output."""
    from deepfilternet_b200 import enhance, init_df, metrics
    g = fixture()
    names = [str(n) for n in g["names"]]
    d3 = np.load(os.path.join(GOLD, "dfnet_DeepFilterNet3.npz"))
    model, st, _, _ = init_df(os.path.join(model_dir, "DeepFilterNet3"), log_level="ERROR")
    audio = torch.from_numpy(d3["audio"])
    out = enhance(model, st, audio)
    r = metrics.evaluate(audio.cuda(), out.cuda(), 48000)
    for ch in range(audio.shape[0]):
        assert_matches([float(r[m][ch]) for m in COLS], g["values"][names.index(f"dfn3_{ch}")], f"dfn3_{ch}")
