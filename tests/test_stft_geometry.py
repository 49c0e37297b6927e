"""STFT geometries other than 960 / 480 (the runtime mixed-radix kernels k_analysis_any / k_apply_synthesis_any): the
host emulation of their FFT and the oracle against the reference modules' outputs at two derived geometries (CPU), and
on the GPU every layer -- libdf, features, DfNet.forward, enhance, chunked and streaming execution, LSNR gating, the
CLI -- against the CPU oracle at 16000/320/160, 48000/480/240 and 44100/882/441, plus the 75 % overlap and
non-divisor hops of the STFT-only interfaces."""
import os
import subprocess

import numpy as np
import pytest
import torch

import dfnet_oracle as O
import libdf_oracle as LO
import random_models
from tests_common import synth_audio

from deepfilternet_b200 import DfNet, _lib, enhance, enhance_device, init_df, libdf
from deepfilternet_b200.config import ModelConfig, load_config
from deepfilternet_b200.enhance import df_features
from deepfilternet_b200.model import find_checkpoint, load_state_dict_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RMS_TOL = 1e-4
TOL_M, TOL_SPEC, TOL_COEF, TOL_LSNR = 1e-5, 1e-6, 1e-5, 1e-3   # as test_gpu_parity.py

GEOS = [(16000, 320, 160), (48000, 480, 240), (44100, 882, 441)]
# STFT-only interfaces also take hops below fft / 2: 75 % overlap, a hop that does not divide fft, a power of two
STFT_GEOS = GEOS + [(48000, 960, 240), (48000, 960, 400), (16000, 512, 256)]
GOLDEN_MODELS = {"DeepFilterNet3_16k": (16000, 320, 160), "DeepFilterNet3_5ms": (48000, 480, 240)}
gid = lambda g: "x".join(map(str, g))


def rms(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.sqrt(((a - b) ** 2).mean()))


def cfg_of(kind, geo):
    sr, fft, hop = geo
    base = dict(conv_ch=64, df_pathway_kernel_size_t=5, sr=sr, fft_size=fft, hop_size=hop)
    if kind == "dfn3":
        return ModelConfig(model="deepfilternet3", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=16, enc_lin_groups=32, df_gru_skip="groupedlinear", **base)
    if kind == "dfn2":
        return ModelConfig(model="deepfilternet2", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=8, enc_lin_groups=8, enc_concat=True, **base)
    if kind == "v1":
        return ModelConfig(model="deepfilternet", conv_lookahead=2, df_lookahead=1, conv_kernel=(2, 3), convt_kernel=(2, 3),
                           conv_kernel_inp=(2, 3), conv_k_enc=2, conv_k_dec=2, emb_hidden_dim=512, df_hidden_dim=512,
                           emb_num_layers=3, df_num_layers=2, gru_groups=8, lin_groups=8, enc_lin_groups=8, group_shuffle=True,
                           dfop_method="real_unfold", **base)
    return ModelConfig(model="deepfilternet3", conv_lookahead=0, df_lookahead=0, conv_kernel=(2, 3), emb_hidden_dim=512,
                       df_hidden_dim=512, emb_num_layers=3, df_num_layers=3, lin_groups=16, enc_lin_groups=16,
                       df_gru_skip="groupedlinear", **base)


def dstate(geo, device_side=True):
    sr, fft, hop = geo
    return libdf.DF(sr, fft, hop, 32, 2) if device_side else LO.DF(sr, fft, hop, 32, 2)


@pytest.fixture(scope="module")
def geo_model_dir(tmp_path_factory):
    """Model directories of the committed derived configs (tests/golden/models/DeepFilterNet3_{16k,5ms}) with the seeded
    DeepFilterNet3 weights -- the ones oracle/gen_golden_geometry.py ran the reference modules with."""
    root = str(tmp_path_factory.mktemp("geo_models"))
    sd = random_models.state_dict("DeepFilterNet3")
    for name in GOLDEN_MODELS:
        d = os.path.join(root, name)
        os.makedirs(os.path.join(d, "checkpoints"))
        with open(os.path.join(random_models.CONFIGS, name, "config.ini")) as f, open(os.path.join(d, "config.ini"), "w") as g:
            g.write(f.read())
        torch.save(sd, os.path.join(d, "checkpoints", random_models.CHECKPOINTS["DeepFilterNet3"]))
    return root


# ================================================================== CPU ====
def test_runtime_fft_host_emulation(tmp_path):
    """The runtime mixed-radix transform (dfb_fft.cuh: Stockham passes of radix 4/2/3/5/7, real split / merge) with the
    32 lanes emulated on the CPU, forward and inverse, against a double-precision DFT: max error <= 1e-5 max|X|."""
    exe = tmp_path / "fft_any_host_test"
    subprocess.check_call(["nvcc", "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", "-o", str(exe),
                           os.path.join(ROOT, "tests", "host", "fft_any_host_test.cu")], stderr=subprocess.DEVNULL)
    sizes = [320, 384, 480, 512, 640, 768, 882, 960, 1024, 1536, 1920, 2048, 4096, 160, 400]
    r = subprocess.run([str(exe)] + [str(n) for n in sizes], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    assert len(r.stdout.splitlines()) == len(sizes)


@pytest.mark.parametrize("name", list(GOLDEN_MODELS))
def test_oracle_matches_reference_modules_at_geometry(name, golden_dir, geo_model_dir):
    """tests/golden/dfnet_<name>.npz were produced by the reference's own DfNet / enhance() (oracle/gen_golden_geometry.py);
    same tolerances as the shipped configs in test_oracle_golden.py."""
    g = np.load(os.path.join(golden_dir, f"dfnet_{name}.npz"))
    d = os.path.join(geo_model_dir, name)
    cfg = load_config(os.path.join(d, "config.ini"), env={})
    assert (cfg.sr, cfg.fft_size, cfg.hop_size) == GOLDEN_MODELS[name]
    sd = load_state_dict_file(find_checkpoint(os.path.join(d, "checkpoints"))[0])
    audio = torch.from_numpy(g["audio"])
    out, aux = O.enhance(sd, cfg.as_dict(), audio, pad=True, return_all=True)
    assert aux["spec"].shape[-2] == cfg.fft_size // 2 + 1
    assert np.abs(aux["spec"].numpy() - g["spec"]).max() < 1e-7
    assert np.abs(aux["erb_feat"].numpy() - g["feat_erb"]).max() < 1e-6
    assert np.abs(aux["spec_feat"].numpy() - g["feat_spec"]).max() < 1e-6
    assert np.abs(aux["m"].numpy() - g["m"]).max() < 1e-5
    assert np.abs(aux["lsnr"].numpy() - g["lsnr"]).max() < 1e-3
    assert np.abs(aux["spec_e"].numpy() - g["spec_e"]).max() < 1e-6
    assert float(np.sqrt(((out.numpy() - g["enhanced"]) ** 2).mean())) < 1e-6
    o2 = O.enhance(sd, cfg.as_dict(), audio, pad=False)
    assert o2.shape == g["enhanced_nopad"].shape
    assert float(np.sqrt(((o2.numpy() - g["enhanced_nopad"]) ** 2).mean())) < 1e-6
    o3 = O.enhance(sd, cfg.as_dict(), audio, pad=True, atten_lim_db=12.0)
    assert float(np.sqrt(((o3.numpy() - g["enhanced_atten12"]) ** 2).mean())) < 1e-6


def test_unsupported_sizes_name_the_rule():
    """fft_size must be even, 32..4096, with no prime factor above 7 in fft_size / 2; checked before any device work."""
    for fft, hop in ((968, 484), (961, 480), (8192, 4096), (16, 8)):
        with pytest.raises(_lib.DfbError, match="no prime factor above 7") as e:
            libdf.DF(48000, fft, hop, 32, 2)
        assert e.value.code == _lib.DFB_ERR_UNSUPPORTED
    with pytest.raises(RuntimeError, match="hop_size \\* 2 <= fft_size"):
        libdf.DF(16000, 320, 161, 32, 2)


# ================================================================== GPU: libdf ====
@pytest.mark.gpu
@pytest.mark.parametrize("geo", STFT_GEOS, ids=gid)
def test_df_analysis_synthesis(geo):
    sr, fft, hop = geo
    st, ost = dstate(geo), dstate(geo, False)
    assert (st.sr(), st.fft_size(), st.hop_size(), st.nb_erb()) == (sr, fft, hop, 32)
    assert st.erb_widths().tolist() == ost.erb_widths().tolist() and int(st.erb_widths().sum()) == fft // 2 + 1
    assert np.array_equal(st.fft_window(), ost.fft_window())
    for C, T in ((1, hop), (1, 7 * hop + hop - 1), (3, 40 * hop + 77), (1, 12345)):
        x = synth_audio(C, T, seed=T, sr=sr).numpy()
        a, b = st.analysis(x), ost.analysis(x)
        assert a.shape == b.shape == (C, T // hop, fft // 2 + 1) and a.dtype == np.complex64
        assert np.abs(a - b).max() < 2e-6, (C, T)
        y, z = st.synthesis(b.copy()), ost.synthesis(b.copy())
        assert y.shape == z.shape == (C, (T // hop) * hop)
        assert np.abs(y - z).max() < 4e-6, (C, T)


@pytest.mark.gpu
@pytest.mark.parametrize("geo", STFT_GEOS, ids=gid)
def test_df_carried_state_and_reconstruction(geo):
    """pyDF reset=False: the fft - hop samples of STFT / ISTFT memory carry from call to call and channel to channel
    (also when a call holds fewer samples than the memory); STFT -> ISTFT reconstructs with delay fft - hop
    (transforms.rs:618-638)."""
    sr, fft, hop = geo
    st, ost = dstate(geo), dstate(geo, False)
    x = synth_audio(3, 30 * hop + 123, seed=5, sr=sr).numpy()
    bounds = [0, 5 * hop, 6 * hop, 6 * hop + 1, 30 * hop + 123]       # incl. a one-frame and a zero-frame call
    for i in range(len(bounds) - 1):
        xa = np.ascontiguousarray(x[:, bounds[i]:bounds[i + 1]])
        a, b = st.analysis(xa, reset=False), ost.analysis(xa, reset=False)
        assert a.shape == b.shape and (a.size == 0 or np.abs(a - b).max() < 2e-6), i
        if b.shape[1]:
            y, z = st.synthesis(b.copy(), reset=False), ost.synthesis(b.copy(), reset=False)
            assert np.abs(y - z).max() < 4e-6, i
    # one channel in chunks == one call over the whole signal
    st.reset()
    whole = st.analysis(x[:1, :24 * hop], reset=True)
    st.reset()
    parts = np.concatenate([st.analysis(np.ascontiguousarray(x[:1, o:o + 4 * hop]), reset=False) for o in range(0, 24 * hop, 4 * hop)], 1)
    assert np.array_equal(whole, parts)
    st.reset()
    xr = synth_audio(2, 200 * hop, seed=3, sr=sr).numpy()
    y = st.synthesis(st.analysis(xr))
    if fft % hop:
        # the squared vorbis window does not sum to a constant at a hop that does not divide fft, so the reference does
        # not reconstruct either (1 - corr = 6e-3 at 960 / 400): same output as the reference instead
        assert np.abs(y - ost.synthesis(ost.analysis(xr))).max() < 4e-6
        return
    d = fft - hop
    for c in range(2):
        a, b = xr[c, :-d], y[c, d:]
        assert float(np.dot(a, b) / np.sqrt(np.dot(a, a) * np.dot(b, b))) > 1 - 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("geo", GEOS, ids=gid)
def test_features_match_oracle_composition(geo):
    from deepfilternet_b200.features import fft_features
    sr, fft, hop = geo
    st, ost = dstate(geo), dstate(geo, False)
    x = synth_audio(3, 60 * hop + 11, seed=7, sr=sr)
    sp, fe, fs = df_features(x, st, 96, alpha=0.99)
    spec = ost.analysis(x.numpy())
    assert np.abs(sp.numpy() - torch.view_as_real(torch.from_numpy(spec)).unsqueeze(1).numpy()).max() < 2e-6
    assert np.abs(fe.numpy()[:, 0] - LO.erb_norm(LO.erb(spec, ost.erb_widths()), 0.99)).max() < 2e-6
    un = LO.unit_norm(np.ascontiguousarray(spec[..., :96]), 0.99)
    assert np.abs(fs.numpy()[:, 0] - np.stack([un.real, un.imag], -1)).max() < 1e-5
    speech = synth_audio(3, 60 * hop + 11, seed=8, sr=sr)
    out = fft_features(st, x.cuda(), speech.cuda(), nb_spec=96, norm_alpha=0.99)
    assert np.abs(out["noisy"].cpu().numpy()[:, 0] - np.stack([spec.real, spec.imag], -1)).max() < 2e-6
    sp2 = ost.analysis(speech.numpy())
    assert np.abs(out["speech"].cpu().numpy()[:, 0] - np.stack([sp2.real, sp2.imag], -1)).max() < 2e-6
    assert np.abs(out["feat_erb"].cpu().numpy()[:, 0] - LO.erb_norm(LO.erb(spec, ost.erb_widths()), 0.99)).max() < 2e-6


# ================================================================== GPU: DfNet / enhance ====
FORWARD_CASES = [("dfn3", g) for g in GEOS] + [("dfn2", GEOS[0]), ("ll", GEOS[0])]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,geo", FORWARD_CASES, ids=lambda v: v if isinstance(v, str) else gid(v))
def test_forward_and_enhance_vs_oracle(kind, geo):
    sr, fft, hop = geo
    st = dstate(geo)
    cfg = cfg_of(kind, geo)
    sd = random_models_sd(cfg, 2)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(3, 50 * hop + 37, seed=21, sr=sr)
    out_o, aux = O.enhance(sd, cfg.as_dict(), audio, return_all=True)
    spec_e, m, lsnr, last = model(aux["spec"], aux["erb_feat"], aux["spec_feat"])
    assert spec_e.shape == aux["spec_e"].shape and spec_e.shape[-2] == fft // 2 + 1
    assert rms(m, aux["m"]) < TOL_M and rms(spec_e, aux["spec_e"]) < TOL_SPEC
    assert np.abs(lsnr.numpy() - aux["lsnr"].numpy()).max() < TOL_LSNR
    if cfg.model == "deepfilternet3":
        assert rms(last.permute(0, 2, 3, 1, 4).reshape(aux["coefs"].shape), aux["coefs"]) < TOL_COEF
    out = enhance(model, st, audio)
    assert out.shape == audio.shape and rms(out, out_o) < RMS_TOL


def random_models_sd(cfg, seed):
    from deepfilternet_b200.weights import random_state_dict
    return random_state_dict(cfg, seed=seed)


@pytest.mark.gpu
def test_forward_at_75_percent_overlap():
    """DfNet.forward (dfb_model_forward_full: DNN + apply kernel writing the enhanced spectrum) takes any hop."""
    geo = (48000, 960, 240)
    st = dstate(geo)
    cfg = cfg_of("dfn3", geo)
    sd = random_models_sd(cfg, 3)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(2, 9600, seed=22)
    _, aux = O.enhance(sd, cfg.as_dict(), audio, return_all=True)
    spec_e, m, lsnr, _ = model(aux["spec"], aux["erb_feat"], aux["spec_feat"])
    assert rms(m, aux["m"]) < TOL_M and rms(spec_e, aux["spec_e"]) < TOL_SPEC
    assert np.abs(lsnr.numpy() - aux["lsnr"].numpy()).max() < TOL_LSNR


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GOLDEN_MODELS))
def test_golden_reference_outputs_at_geometry(name, golden_dir, geo_model_dir):
    g = np.load(os.path.join(golden_dir, f"dfnet_{name}.npz"))
    model, st, suffix, _ = init_df(os.path.join(geo_model_dir, name), log_level="ERROR")
    assert suffix == name and (st.sr(), st.fft_size(), st.hop_size()) == GOLDEN_MODELS[name]
    audio = torch.from_numpy(g["audio"])
    assert rms(enhance(model, st, audio), g["enhanced"]) < RMS_TOL
    o = enhance(model, st, audio, pad=False)
    assert o.shape == g["enhanced_nopad"].shape and rms(o, g["enhanced_nopad"]) < RMS_TOL
    assert rms(enhance(model, st, audio, atten_lim_db=12.0), g["enhanced_atten12"]) < RMS_TOL
    spec_e, m, lsnr, _ = model(torch.from_numpy(g["spec"]), torch.from_numpy(g["feat_erb"]), torch.from_numpy(g["feat_spec"]))
    assert rms(spec_e, g["spec_e"]) < TOL_SPEC and rms(m, g["m"]) < TOL_M and np.abs(lsnr.numpy() - g["lsnr"]).max() < TOL_LSNR
    assert rms(enhance(model, st, audio), O.enhance(model.state_dict(), model.cfg.as_dict(), audio)) < RMS_TOL


@pytest.mark.gpu
def test_post_filter_mask_only_and_v1_at_16k():
    import dfnet1_oracle as O1
    geo = GEOS[0]
    st = dstate(geo)
    audio = synth_audio(2, 8000, seed=33, sr=16000)
    for kind in ("dfn3", "dfn2"):
        cfg = cfg_of(kind, geo)
        sd = random_models_sd(cfg, 4)
        for opt in ("mask_pf", "mask_only"):
            c = cfg_of(kind, geo)
            setattr(c, opt, True)
            model = DfNet(c, sd, st, run_df=opt != "mask_only")
            ref = O.enhance(sd, dict(cfg.as_dict(), **{opt: True}), audio)
            assert rms(enhance(model, st, audio), ref) < RMS_TOL, (kind, opt)
            assert rms(ref, O.enhance(sd, cfg.as_dict(), audio)) > 1e-5, (kind, opt)   # not a no-op
    cfg = cfg_of("v1", geo)
    sd = random_models_sd(cfg, 7)
    model = DfNet(cfg, sd, st)
    ocfg = dict(O1.DEFAULTS_DFN1, sr=16000, fft_size=320, hop_size=160)
    out_o, aux = O1.enhance(sd, ocfg, audio, return_all=True)
    spec_e, m, lsnr, alpha = model(aux["spec"], aux["erb_feat"], aux["spec_feat"])
    assert rms(m, aux["m"]) < TOL_M and rms(spec_e, aux["spec_e"]) < TOL_SPEC
    assert np.abs(alpha.numpy() - aux["alpha"].numpy()).max() < 1e-4
    assert rms(enhance(model, st, audio), out_o) < RMS_TOL


@pytest.mark.gpu
def test_streams_independent_at_16k():
    geo = GEOS[0]
    st = dstate(geo)
    cfg = cfg_of("dfn3", geo)
    model = DfNet(cfg, random_models_sd(cfg, 4), st)
    audio = synth_audio(12, 16000, seed=31, sr=16000).cuda()
    full = enhance_device(model, st, audio)
    single = enhance_device(model, st, audio[7:8].contiguous())
    perm = torch.randperm(12, generator=torch.Generator().manual_seed(0)).cuda()
    shuffled = enhance_device(model, st, audio[perm].contiguous())
    torch.cuda.synchronize()
    assert rms(full[7:8].cpu(), single.cpu()) < 1e-7 and rms(full[perm].cpu(), shuffled.cpu()) < 1e-7


CHUNK_CASES = [("dfn3", GEOS[0]), ("dfn2", GEOS[0]), ("dfn3", GEOS[1])]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,geo", CHUNK_CASES, ids=lambda v: v if isinstance(v, str) else gid(v))
def test_chunked_and_streaming_equal_one_shot(kind, geo):
    from deepfilternet_b200 import DfStream
    sr, fft, hop = geo
    st = dstate(geo)
    cfg = cfg_of(kind, geo)
    sd = random_models_sd(cfg, 13)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(3, 400 * hop + 57, seed=61, sr=sr, device="cuda")
    model.set_chunking(1, 1, 1)
    one = enhance_device(model, st, audio).clone()
    model.set_chunking(6, 6, 2)
    six = enhance_device(model, st, audio).clone()
    host = enhance(model, st, audio.cpu())
    torch.cuda.synchronize()
    assert rms(one.cpu(), six.cpu()) < 1e-6 and rms(one.cpu(), host) < 1e-6
    assert rms(one.cpu(), O.enhance(sd, cfg.as_dict(), audio.cpu())) < RMS_TOL
    model.set_chunking()
    n = 157
    x = audio[:2, :n * hop].cpu().contiguous()
    ref = enhance(model, st, x, pad=False)
    s = DfStream(model, st, batch=2)
    assert s.hop == hop
    outs, pos = [], 0
    for i, k in enumerate([1, 1, 2, 1, 7, 40, 1, 3, 64, 30, 7]):
        outs.append(s.process(x[:, pos * hop:(pos + k) * hop].cuda() if i % 2 else x[:, pos * hop:(pos + k) * hop]).cpu())
        pos += k
    outs.append(s.flush())
    got = torch.cat(outs, 1)
    lat = s.latency_frames * hop
    assert got.shape == (2, n * hop + lat) and (lat == 0 or got[:, :lat].abs().max() == 0)
    assert rms(got[:, lat:], ref) < 1e-6


@pytest.mark.gpu
def test_streaming_lsnr_stage_gating_at_16k():
    """tract.rs:658-672 stage semantics on k_apply_synthesis_any, checked by definition as in test_gpu_parity.py."""
    from deepfilternet_b200 import DfStream
    geo = GEOS[0]
    st = dstate(geo)
    cfg = cfg_of("dfn3", geo)
    sd = random_models_sd(cfg, 15)
    model = DfNet(cfg, sd, st)
    hop, n = 160, 90
    audio = synth_audio(2, hop * n, seed=81, sr=16000)

    def run(model, **th):
        s = DfStream(model, st, batch=2, atten_lim_db=th.pop("atten", None))
        if th:
            s.set_lsnr_thresholds(**th)
        return torch.cat([s.process(audio[:, :hop * 33]), s.process(audio[:, hop * 33:]), s.flush()], 1)[:, s.latency_frames * hop:]

    base = run(model)
    assert rms(run(model, min_db_thresh=-1e9, max_db_erb_thresh=1e9, max_db_df_thresh=1e9), base) < 1e-7
    gains_only = run(model, min_db_thresh=-1e9, max_db_erb_thresh=1e9, max_db_df_thresh=-1e9)
    assert rms(gains_only, run(DfNet(cfg, sd, st, run_df=False))) < 1e-7 and rms(gains_only, base) > 1e-5
    passthrough = run(model, min_db_thresh=-1e9, max_db_erb_thresh=-1e9, max_db_df_thresh=-1e9)
    ident = torch.from_numpy(st.synthesis(st.analysis(audio.numpy())))
    assert rms(passthrough, ident) < 1e-6
    assert run(model, min_db_thresh=1e9, max_db_erb_thresh=2e9, max_db_df_thresh=2e9).abs().max() < 1e-7
    z = run(model, min_db_thresh=1e9, max_db_erb_thresh=2e9, max_db_df_thresh=2e9, atten=12.0)
    assert rms(z, ident * 10 ** (-12 / 20)) < 1e-6


@pytest.mark.gpu
def test_cli_resamples_through_a_16k_model(tmp_path, golden_dir, geo_model_dir):
    """`deepFilter` with the 16 kHz model on a 48 kHz file: resampled to 16 kHz, enhanced, resampled back to 48 kHz."""
    from deepfilternet_b200 import io as dio
    from deepfilternet_b200.enhance import run
    src = os.path.join(golden_dir, "assets", "noisy_snr0.wav")
    audio, meta = dio.load_audio(src, 48000)
    out_dir = tmp_path / "out"
    assert run(["-m", os.path.join(geo_model_dir, "DeepFilterNet3_16k"), "-o", str(out_dir), "--log-level", "ERROR", src]) == 0
    written, wmeta = dio.load_audio(str(out_dir / "noisy_snr0_DeepFilterNet3_16k.wav"))
    model, st, _, _ = init_df(os.path.join(geo_model_dir, "DeepFilterNet3_16k"), log_level="ERROR")
    ref = dio.resample(enhance(model, st, dio.resample(audio, 48000, 16000)), 16000, 48000)
    ref = (ref * (1 << 15)).to(torch.int16).to(torch.float32) / 32768.0
    # like the reference (enhance.py:88-89) the output is not trimmed: the input length up to the rounding of the
    # 48 -> 16 -> 48 kHz round trip
    assert wmeta.sample_rate == 48000 and written.shape == ref.shape and abs(written.shape[1] - audio.shape[1]) <= 3
    assert float((written - ref).abs().max()) <= 1.0 / 32768.0 + 1e-7


@pytest.mark.gpu
def test_geometry_errors():
    cfg = cfg_of("dfn3", (48000, 960, 240))
    st = dstate((48000, 960, 240))
    model = DfNet(cfg, random_models_sd(cfg, 1), st)
    with pytest.raises(_lib.DfbError, match="hop_size == fft_size / 2") as e:
        enhance(model, st, synth_audio(1, 4800, seed=1))
    assert e.value.code == _lib.DFB_ERR_UNSUPPORTED
    from deepfilternet_b200 import DfStream
    with pytest.raises(_lib.DfbError, match="hop_size == fft_size / 2") as e:
        DfStream(model, st, batch=1)
    assert e.value.code == _lib.DFB_ERR_UNSUPPORTED
    small = (16000, 128, 64)                           # F = 65 < nb_df = 96
    cfg = cfg_of("dfn3", small)
    with pytest.raises(_lib.DfbError, match="exceeds the 65 frequency bins") as e:
        DfNet(cfg, random_models_sd(cfg, 1), dstate(small))
    assert e.value.code == _lib.DFB_ERR_INVALID


def _kernel_names():
    import ctypes
    buf = ctypes.create_string_buffer(1 << 16)
    n = _lib.lib().dfb_profile_report(buf, len(buf))
    assert n >= 0
    return {line.split()[0] for line in buf.value.decode().splitlines() if line}


@pytest.mark.gpu
def test_dispatch_by_geometry():
    """960 / 480 runs the specialised kernels only; any other geometry the runtime mixed-radix ones."""
    lib = _lib.lib()
    try:
        for geo, want, avoid in (((48000, 960, 480), {"k_analysis", "k_apply_synthesis"}, {"k_analysis_any", "k_apply_synthesis_any"}),
                                 ((16000, 320, 160), {"k_analysis_any", "k_apply_synthesis_any"}, {"k_analysis", "k_apply_synthesis"})):
            st = dstate(geo)
            cfg = cfg_of("dfn3", geo)
            model = DfNet(cfg, random_models_sd(cfg, 1), st)
            torch.cuda.synchronize()
            _kernel_names()
            lib.dfb_profile_enable(1, None)
            enhance(model, st, synth_audio(2, 40 * geo[2], seed=1, sr=geo[0]))
            names = _kernel_names()
            lib.dfb_profile_enable(0, None)
            assert want <= names and not (avoid & names), (geo, names)
    finally:
        lib.dfb_profile_enable(0, None)
        _kernel_names()
