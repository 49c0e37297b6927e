"""GPU: the CUDA path (through the C ABI / its Python mirror) against the CPU oracle on the same
seeded inputs, against the committed golden fixtures, and through size-independent properties at
larger sizes.  Tolerances: integer indexing (ERB widths, frame counts, crop offsets) bit exact;
floating point RMS(out - oracle) <= 1e-4 as BASELINE.json states (measured: ~2e-8)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import dfnet_oracle as O
import libdf_oracle as LO
from tests_common import synth_audio

from deepfilternet_b200 import DfNet, _lib, enhance, enhance_device, init_df, libdf
from deepfilternet_b200.config import ModelConfig, load_config
from deepfilternet_b200.enhance import df_features
from deepfilternet_b200.model import find_checkpoint, load_state_dict_file
from deepfilternet_b200.weights import random_state_dict

RMS_TOL = 1e-4  # BASELINE.json north_star
# tolerances on the intermediate tensors of DfNet.forward (the default arithmetic is BF16x3 on the tensor cores)
TOL_M, TOL_SPEC, TOL_COEF, TOL_LSNR = 1e-5, 1e-6, 1e-5, 1e-3


def rms(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.sqrt(((a - b) ** 2).mean()))


def cfg_of(kind):
    base = dict(conv_ch=64, df_pathway_kernel_size_t=5)
    if kind == "dfn3":
        return ModelConfig(model="deepfilternet3", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=16, enc_lin_groups=32, df_gru_skip="groupedlinear", **base)
    if kind == "dfn2":
        return ModelConfig(model="deepfilternet2", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=8, enc_lin_groups=8, enc_concat=True, **base)
    return ModelConfig(model="deepfilternet3", conv_lookahead=0, df_lookahead=0, conv_kernel=(2, 3), emb_hidden_dim=512,
                       df_hidden_dim=512, emb_num_layers=3, df_num_layers=3, lin_groups=16, enc_lin_groups=16,
                       df_gru_skip="groupedlinear", **base)


@pytest.fixture(scope="module")
def states():
    return libdf.DF(48000, 960, 480, 32, 2), LO.DF(48000, 960, 480, 32, 2)


# ------------------------------------------------------------------ libdf (pyDF boundary) ----
def test_df_accessors(states):
    st, ost = states
    assert st.erb_widths().dtype == np.uint64 and st.erb_widths().tolist() == ost.erb_widths().tolist()
    assert np.array_equal(st.fft_window(), ost.fft_window())
    assert (st.sr(), st.fft_size(), st.hop_size(), st.nb_erb()) == (48000, 960, 480, 32)


@pytest.mark.parametrize("C,T", [(1, 480), (1, 479 + 480), (3, 12345), (2, 48000)])
def test_analysis_synthesis(states, C, T):
    st, ost = states
    x = synth_audio(C, T, seed=11).numpy()
    a, b = st.analysis(x), ost.analysis(x)
    assert a.shape == b.shape == (C, T // 480, 481) and a.dtype == np.complex64
    assert np.abs(a - b).max() < 1e-6
    y, z = st.synthesis(b.copy()), ost.synthesis(b.copy())
    assert y.shape == z.shape == (C, (T // 480) * 480)
    assert np.abs(y - z).max() < 2e-6


def test_analysis_synthesis_carried_state(states):
    """pyDF `reset=False` (pyDF/src/lib.rs:56-58, 91-93): the shared DFState carries the STFT / ISTFT memories
    from call to call and from channel c to channel c + 1; `DF.reset()` clears them."""
    st, ost = states
    st.reset(), ost.reset()
    x = synth_audio(3, 9600 + 123, seed=5).numpy()
    for i, (lo, hi) in enumerate([(0, 2400), (2400, 2880), (2880, 9723)]):   # chunked streaming incl. a 1-frame call
        xa = np.ascontiguousarray(x[:, lo:hi])
        a, b = st.analysis(xa, reset=False), ost.analysis(xa, reset=False)
        assert np.abs(a - b).max() < 1e-6, i
        y, z = st.synthesis(b.copy(), reset=False), ost.synthesis(b.copy(), reset=False)
        assert np.abs(y - z).max() < 2e-6, i
    # a reset=True call still leaves the last channel's memory behind for a following reset=False call
    a, b = st.analysis(x, reset=True), ost.analysis(x, reset=True)
    y, z = st.synthesis(b.copy(), reset=True), ost.synthesis(b.copy(), reset=True)
    x2 = synth_audio(1, 4800, seed=6).numpy()
    a, b = st.analysis(x2, reset=False), ost.analysis(x2, reset=False)
    assert np.abs(a - b).max() < 1e-6
    y, z = st.synthesis(b.copy(), reset=False), ost.synthesis(b.copy(), reset=False)
    assert np.abs(y - z).max() < 2e-6
    # single-channel streaming in chunks == one reset call over the whole signal
    st.reset()
    whole = st.analysis(x[:1, :9600], reset=True)
    st.reset()
    parts = np.concatenate([st.analysis(np.ascontiguousarray(x[:1, o:o + 1920]), reset=False) for o in range(0, 9600, 1920)], 1)
    assert np.array_equal(whole, parts)
    st.reset(), ost.reset()
    assert np.abs(st.analysis(x2, reset=False) - ost.analysis(x2, reset=False)).max() < 1e-6
    st.reset(), ost.reset()


def test_analysis_errors(states):
    st, _ = states
    with pytest.raises(RuntimeError, match="empty or not contiguous"):
        st.analysis(np.zeros((2, 9600), np.float32)[:, ::2])
    with pytest.raises(RuntimeError, match="empty or not contiguous"):
        st.analysis(np.zeros((0, 960), np.float32))
    assert st.analysis(np.zeros((2, 100), np.float32)).shape == (2, 0, 481)  # shorter than one hop
    with pytest.raises(RuntimeError):
        libdf.DF(48000, 960, 500, 32, 2)  # hop * 2 > fft (libDF/src/lib.rs:111)


def test_stft_istft_reconstruction(states):
    """libDF/src/transforms.rs:618-638 on the GPU kernels."""
    st, _ = states
    x = synth_audio(2, 96000, seed=3).numpy()
    y = st.synthesis(st.analysis(x))
    d = 480
    for c in range(2):
        a, b = x[c, :-d], y[c, d:]
        corr = float(np.dot(a, b) / np.sqrt(np.dot(a, a) * np.dot(b, b)))
        assert corr > 1 - 1e-6


def test_erb_family(states):
    st, ost = states
    rng = np.random.default_rng(0)
    spec = (rng.standard_normal((2, 50, 481)) + 1j * rng.standard_normal((2, 50, 481))).astype(np.complex64) * 0.01
    w = st.erb_widths()
    for db in (True, False):
        a, b = libdf.erb(spec, w, db), LO.erb(spec, w, db)
        assert a.shape == (2, 50, 32) and np.allclose(a, b, rtol=1e-5, atol=2e-5)
    assert libdf.erb(spec[0], w).shape == (50, 32) and libdf.erb(spec[None], w).shape == (1, 2, 50, 32)
    with pytest.raises(ValueError, match="Dimension not supported for erb"):
        libdf.erb(spec[0, 0], w)
    e = LO.erb(spec, w)
    assert np.array_equal(libdf.erb_norm(e, 0.99), LO.erb_norm(e, 0.99))
    s0 = rng.standard_normal((2, 32)).astype(np.float32)
    assert np.array_equal(libdf.erb_norm(e, 0.9, s0), LO.erb_norm(e, 0.9, s0))
    assert np.abs(libdf.unit_norm(spec[..., :96].copy(), 0.99) - LO.unit_norm(spec[..., :96].copy(), 0.99)).max() < 1e-5
    u0 = np.abs(rng.standard_normal((2, 481))).astype(np.float32) + 0.01
    assert np.abs(libdf.unit_norm(spec, 0.95, u0) - LO.unit_norm(spec, 0.95, u0)).max() < 1e-5
    assert np.array_equal(libdf.unit_norm_init(96), LO.unit_norm_init(96))
    g = rng.uniform(0, 1, (2, 7, 32)).astype(np.float32)
    assert np.array_equal(libdf.erb_inv(g, w), LO.erb_inv(g, w))
    with pytest.raises(ValueError, match="Number of erb bands do not match"):
        libdf.erb_inv(g[..., :31], w)


def test_df_features_matches_reference_composition(states):
    """df_features (enhance.py:190-203) == analysis -> erb -> erb_norm / unit_norm, one fused pass."""
    st, ost = states
    x = synth_audio(3, 24000, seed=7)
    sp, fe, fs = df_features(x, st, 96, alpha=0.99)
    spec = ost.analysis(x.numpy())
    assert np.abs(sp.numpy() - torch.view_as_real(torch.from_numpy(spec)).unsqueeze(1).numpy()).max() < 1e-6
    assert np.abs(fe.numpy()[:, 0] - LO.erb_norm(LO.erb(spec, ost.erb_widths()), 0.99)).max() < 2e-6
    ref = torch.view_as_real(torch.from_numpy(LO.unit_norm(np.ascontiguousarray(spec[..., :96]), 0.99))).unsqueeze(1)
    assert np.abs(fs.numpy() - ref.numpy()).max() < 1e-5


# ------------------------------------------------------------------ DfNet.forward ----
@pytest.mark.parametrize("kind,B,T", [("dfn3", 3, 24000), ("dfn3", 1, 4800), ("dfn2", 2, 19200), ("ll", 5, 14400),
                                      ("dfn3", 9, 9600), ("ll", 17, 4800)])
def test_forward_random_weights(states, kind, B, T):
    st, _ = states
    cfg = cfg_of(kind)
    sd = random_state_dict(cfg, seed=2)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(B, T, seed=21)
    out_o, aux = O.enhance(sd, cfg.as_dict(), audio, return_all=True)
    spec_e, m, lsnr, last = model(aux["spec"], aux["erb_feat"], aux["spec_feat"])
    assert spec_e.shape == aux["spec_e"].shape and m.shape == aux["m"].shape and lsnr.shape == aux["lsnr"].shape
    assert rms(m, aux["m"]) < TOL_M and rms(spec_e, aux["spec_e"]) < TOL_SPEC
    assert np.abs(lsnr.numpy() - aux["lsnr"].numpy()).max() < TOL_LSNR
    if cfg.model == "deepfilternet3":
        assert last.shape == (B, 5, aux["m"].shape[2], 96, 2)
        assert rms(last.permute(0, 2, 3, 1, 4).reshape(aux["coefs"].shape), aux["coefs"]) < TOL_COEF
    out = enhance(model, st, audio)
    assert out.shape == audio.shape and rms(out, out_o) < RMS_TOL
    # CUDA-tensor in, CUDA-tensor out through the same forward
    r = model(aux["spec"].cuda(), aux["erb_feat"].cuda(), aux["spec_feat"].cuda())
    assert r[0].is_cuda and rms(r[0].cpu(), aux["spec_e"]) < TOL_SPEC


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_golden_reference_outputs(name, golden_dir, model_dir):
    """Against outputs of the reference's own modules (tests/golden, made by oracle/gen_golden.py)."""
    g = np.load(os.path.join(golden_dir, f"dfnet_{name}.npz"))
    model, st, suffix, epoch = init_df(os.path.join(model_dir, name), log_level="ERROR")
    assert suffix == name
    audio = torch.from_numpy(g["audio"])
    assert rms(enhance(model, st, audio), g["enhanced"]) < RMS_TOL
    o = enhance(model, st, audio, pad=False)
    assert o.shape == g["enhanced_nopad"].shape and rms(o, g["enhanced_nopad"]) < RMS_TOL
    assert rms(enhance(model, st, audio, atten_lim_db=12.0), g["enhanced_atten12"]) < RMS_TOL
    spec_e, m, lsnr, _ = model(torch.from_numpy(g["spec"]), torch.from_numpy(g["feat_erb"]), torch.from_numpy(g["feat_spec"]))
    assert rms(spec_e, g["spec_e"]) < TOL_SPEC and rms(m, g["m"]) < TOL_M and np.abs(lsnr.numpy() - g["lsnr"]).max() < TOL_LSNR


def test_ll_model_end_to_end(golden_dir, model_dir):
    """DeepFilterNet3_ll (H = 512, zero look-ahead, kt = 2 convs): init_df on its model directory, against the
    reference modules' outputs with the same weights."""
    g = np.load(os.path.join(golden_dir, "dfnet_DeepFilterNet3_ll.npz"))
    model, st, suffix, epoch = init_df(os.path.join(model_dir, "DeepFilterNet3_ll"), log_level="ERROR")
    assert (model.cfg.conv_lookahead, model.cfg.df_lookahead, model.cfg.emb_hidden_dim) == (0, 0, 512)
    assert rms(enhance(model, st, torch.from_numpy(g["audio"])), g["enhanced"]) < RMS_TOL
    spec_e, m, lsnr, _ = model(torch.from_numpy(g["spec"]), torch.from_numpy(g["feat_erb"]), torch.from_numpy(g["feat_spec"]))
    assert rms(spec_e, g["spec_e"]) < TOL_SPEC and rms(m, g["m"]) < TOL_M


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_si_sdr_known_answer_gpu(name, golden_dir, model_dir):
    """The reference CI's known answer check (df/scripts/test_df.py:44-78, atol = rtol = 1e-4) on the CUDA path, against
    the reference modules' value for the weights of model_dir."""
    import ref_harness as rh
    kat = json.load(open(os.path.join(golden_dir, "kat.json")))[name]
    model, st, _, epoch = init_df(os.path.join(model_dir, name), log_level="ERROR")
    assert epoch == kat["epoch"]
    noisy = torch.from_numpy(rh.read_wav(os.path.join(golden_dir, "assets", "noisy_snr0.wav")))
    clean = rh.read_wav(os.path.join(golden_dir, "assets", "clean_freesound_33711.wav"))
    out = enhance(model, st, noisy, pad=True)
    s = rh.si_sdr(clean, out.numpy())
    assert abs(s - kat["target"]) <= 1e-4 + 1e-4 * abs(kat["target"]), (s, kat["target"])


# ------------------------------------------------------------------ enhance(): properties at size ----
def test_enhance_streams_are_independent_and_batched_equals_single(states):
    """Per-channel state reset (pyDF/src/lib.rs:56-58): a stream's output does not depend on its
    batch neighbours or its position in the batch (covers the GRU cluster grouping and the
    stream-group chunking of dfb_enhance)."""
    st, _ = states
    cfg = cfg_of("dfn3")
    model = DfNet(cfg, random_state_dict(cfg, seed=4), st)
    audio = synth_audio(40, 48000, seed=31).cuda()
    full = enhance_device(model, st, audio)
    perm = torch.randperm(40, generator=torch.Generator().manual_seed(0)).cuda()
    shuffled = enhance_device(model, st, audio[perm].contiguous())
    assert torch.equal(full[perm], shuffled) or rms(full[perm].cpu(), shuffled.cpu()) < 1e-7
    single = enhance_device(model, st, audio[7:8].contiguous())
    assert rms(full[7:8].cpu(), single.cpu()) < 1e-7
    torch.cuda.synchronize()


def test_enhance_full_size_properties(states):
    """BASELINE configs[1] shape per stream (10 s) at reduced batch: finite output, exact length,
    silence in -> silence out, and the oracle on a sample of the streams."""
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=5)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(16, 480000, seed=41)
    audio[3] = 0.0
    out = enhance(model, st, audio)
    assert out.shape == audio.shape and torch.isfinite(out).all()
    assert out[3].abs().max() < 1e-6
    ref = O.enhance(sd, cfg.as_dict(), audio[5:6])
    assert rms(out[5:6], ref) < RMS_TOL


def test_enhance_edge_lengths(states):
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=6)
    model = DfNet(cfg, sd, st)
    for T in (1, 479, 480, 481, 1000, 4801):
        audio = synth_audio(2, T, seed=T)
        out = enhance(model, st, audio)
        assert out.shape == (2, T)
        assert rms(out, O.enhance(sd, cfg.as_dict(), audio)) < RMS_TOL
    with pytest.raises(RuntimeError):
        enhance(model, st, torch.zeros(1, 100), pad=False)  # shorter than one hop without padding


def test_launch_counter_counts_own_kernels(states):
    st, _ = states
    n0 = _lib.lib().dfb_kernel_launches()
    st.analysis(np.zeros((1, 4800), np.float32))
    assert _lib.lib().dfb_kernel_launches() == n0 + 1


@pytest.mark.parametrize("kind", ["dfn3", "dfn2", "ll"])
def test_precision_modes_agree_with_oracle(states, kind):
    """Every arithmetic mode of the contractions (FFMA everywhere ... BF16x3 tcgen05 for the recurrence, the GRU
    projections and the separable conv blocks incl. the fused mask head) stays inside the 1e-4 bound; the
    tensor-core modes must also agree with the all-FFMA mode to ~1e-6."""
    st, _ = states
    cfg = cfg_of(kind)
    sd = random_state_dict(cfg, seed=9)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(3, 14400, seed=31)
    ref = O.enhance(sd, cfg.as_dict(), audio)
    outs = {}
    for mode in ("fp32", "fp32+gru_tc", "fp32+gru_tc+proj_tc", "fp32+gru_tc+proj_tc+conv_tc"):
        model.set_precision(mode)
        outs[mode] = enhance(model, st, audio)
        assert rms(outs[mode], ref) < RMS_TOL, mode
    for mode, o in outs.items():
        assert rms(o, outs["fp32"]) < 5e-6, mode


def test_wide_batch_matches_oracle(states):
    """More than 64 streams: the DF decoder's recurrence switches to 32 streams per cluster and the batched
    kernels run with ragged last tiles; a few of the streams are checked against the oracle."""
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=12)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(70, 7200, seed=41)
    out = enhance(model, st, audio)
    assert out.shape == audio.shape
    for i in (0, 17, 33, 64, 69):  # both halves of a 32-stream cluster, the ragged last cluster
        assert rms(out[i:i + 1], O.enhance(sd, cfg.as_dict(), audio[i:i + 1])) < RMS_TOL, i


# ------------------------------------------------------------------ BASELINE configs at size ----
def _model_dir_weights(name, model_dir_path):
    """(cfg, state_dict) of a model directory laid out like the shipped ones."""
    p = os.path.join(model_dir_path, name)
    cfg = load_config(os.path.join(p, "config.ini"), env={})
    cp, _ = find_checkpoint(os.path.join(p, "checkpoints"))
    return cfg, load_state_dict_file(cp)


@pytest.mark.parametrize("name,kind,B,seconds,rows", [
    ("DeepFilterNet3", "dfn3", 128, 10, (0, 37, 90, 127)),     # cfg2: k_gru_tc<32> (DF decoder) over 1002 steps
    ("DeepFilterNet2", "dfn2", 512, 10, (0, 200, 511)),        # cfg3
    ("DeepFilterNet3_ll", "ll", 256, 10, (3, 255)),            # cfg4 per-GPU shard: H = 512 GRUs, kt = 2 convs
    ("DeepFilterNet3", "dfn3", 24, 30, (5, 23)),               # cfg5 stream length: 3002 frames of state integration
])
def test_baseline_configs_at_size(states, model_dir, name, kind, B, seconds, rows):
    """SURVEY 8d "parity gate on every config": the CUDA path at the BASELINE batch shapes against the oracle on a
    sample of the streams (the oracle needs seconds per stream), plus finiteness / exact length of the whole batch."""
    st, _ = states
    if name == "DeepFilterNet3_ll":
        cfg = cfg_of("ll")
        sd = random_state_dict(cfg, seed=3)
    else:
        cfg, sd = _model_dir_weights(name, model_dir)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(B, 48000 * seconds, seed=77, device="cuda")
    out = enhance_device(model, st, audio)
    torch.cuda.synchronize()
    assert out.shape == audio.shape and torch.isfinite(out).all()
    idx = list(rows)
    ref = O.enhance(sd, cfg.as_dict(), audio[idx].cpu())
    got = out[idx].cpu()
    for j, i in enumerate(idx):
        assert rms(got[j], ref[j]) < RMS_TOL, (name, i, rms(got[j], ref[j]))


def test_stream_groups_with_ragged_last_group(states):
    """When not even a short time chunk of the whole batch fits the workspace cap, dfb_enhance also splits the batch into
    stream groups: force small groups (of 43 streams, with a ragged last group) with several time chunks each and require the
    same output as the uncapped run, and the oracle on streams of several groups."""
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=8)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(43, 48000, seed=51, device="cuda")
    full = enhance_device(model, st, audio).clone()
    torch.cuda.synchronize()
    per_stream = model.workspace_bytes() / 43
    model.set_max_workspace(int(per_stream * 3.2))
    grouped = enhance_device(model, st, audio)
    torch.cuda.synchronize()
    assert torch.equal(full, grouped) or rms(full.cpu(), grouped.cpu()) < 1e-6
    host = enhance(model, st, audio.cpu())          # the host entry point takes the same grouped route
    assert rms(host, full.cpu()) < 1e-6
    for i in (0, 4, 5, 22, 39, 42):
        assert rms(grouped[i:i + 1].cpu(), O.enhance(sd, cfg.as_dict(), audio[i:i + 1].cpu())) < RMS_TOL, i
    model.set_max_workspace(64 << 30)


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_whole_asset_rms_against_oracle(name, golden_dir, model_dir):
    """The whole 10.6 s reference recording: RMS(out - oracle) <= 1e-4 (the SI-SDR KAT above
    is a scalar with 1e-4 relative slack; this compares every sample)."""
    import ref_harness as rh
    model, st, _, _ = init_df(os.path.join(model_dir, name), log_level="ERROR")
    noisy = torch.from_numpy(rh.read_wav(os.path.join(golden_dir, "assets", "noisy_snr0.wav")))
    out = enhance(model, st, noisy, pad=True)
    ref = O.enhance(model.state_dict(), model.cfg.as_dict(), noisy)
    assert out.shape == ref.shape and rms(out, ref) < RMS_TOL


def test_mismatched_df_state_is_rejected(states):
    """A DF state with another band layout than the model's must be refused, not indexed out of bounds (ADVICE r1)."""
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=1)
    with pytest.raises(ValueError):
        DfNet(cfg, sd, libdf.DF(48000, 960, 480, 24, 2))
    model = DfNet(cfg, sd, st)
    other = libdf.DF(48000, 960, 480, 32, 1)      # same band count, different widths (min_nb_erb_freqs = 1)
    with pytest.raises(RuntimeError):
        enhance(model, other, synth_audio(1, 4800, seed=1))
    with pytest.raises(ValueError):
        enhance_device(model, st, synth_audio(2, 4800, seed=1).cuda(), out=torch.empty(2, 100, device="cuda"))


# ------------------------------------------------------------------ time chunks / streaming ----
@pytest.mark.parametrize("kind", ["dfn3", "dfn2", "ll"])
def test_time_chunked_enhance_equals_one_shot(states, kind):
    """dfb_enhance runs in time chunks with carried state (STFT / ISTFT memories, norm EMAs, GRU states, conv and deep
    filter history -- SURVEY Appendix D).  One chunk, six chunks back to back, six chunks pipelined over the two lanes
    (encoder of chunk c + 1 overlapping the decoder of chunk c) and a workspace cap that forces many short chunks must all
    give the same audio, on the device and the host path, and match the oracle."""
    st, _ = states
    cfg = cfg_of(kind)
    sd = random_state_dict(cfg, seed=13)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(3, 48000 * 5 + 123, seed=61, device="cuda")    # 501 frames + a partial hop
    model.set_chunking(1, 1, 1)
    one = enhance_device(model, st, audio).clone()
    torch.cuda.synchronize()
    per_stream = model.workspace_bytes() / 3
    model.set_chunking(6, 6, 1)
    serial6 = enhance_device(model, st, audio).clone()
    model.set_chunking(6, 6, 2)
    piped = enhance_device(model, st, audio).clone()
    piped2 = enhance_device(model, st, audio).clone()                  # back to back: lanes are reused correctly
    host = enhance(model, st, audio.cpu())
    nopad = enhance_device(model, st, audio, pad=False).clone()
    model.set_max_workspace(int(per_stream * 3 * 2 * 60 / 503))        # ~ 50-frame windows on each lane
    many = enhance_device(model, st, audio).clone()
    many_host = enhance(model, st, audio.cpu())
    torch.cuda.synchronize()
    model.set_max_workspace(64 << 30)
    for name, x in (("serial6", serial6), ("piped", piped), ("piped2", piped2), ("many", many)):
        assert rms(one.cpu(), x.cpu()) < 1e-6, name
    assert rms(one.cpu(), host) < 1e-6 and rms(one.cpu(), many_host) < 1e-6
    ref = O.enhance(sd, cfg.as_dict(), audio.cpu())
    assert rms(many.cpu(), ref) < RMS_TOL and rms(piped.cpu(), ref) < RMS_TOL
    assert rms(nopad.cpu(), O.enhance(sd, cfg.as_dict(), audio.cpu(), pad=False)) < RMS_TOL


@pytest.mark.parametrize("kind", ["dfn3", "dfn2", "ll"])
def test_streaming_equals_one_shot(states, kind):
    """SURVEY 8(f)-1: frame-incremental processing (DfTract::process, tract.rs:509-642) == one-shot enhance(pad=False)
    delayed by the model's look-ahead, for ragged call sizes down to a single hop, device and host tensors."""
    from deepfilternet_b200 import DfStream
    st, _ = states
    cfg = cfg_of(kind)
    sd = random_state_dict(cfg, seed=14)
    model = DfNet(cfg, sd, st)
    hop, n = 480, 157
    audio = synth_audio(2, hop * n, seed=71)
    ref = enhance(model, st, audio, pad=False)            # [2, n * hop], delayed by fft - hop
    s = DfStream(model, st, batch=2)
    assert s.hop == hop and s.latency_frames == max(cfg.conv_lookahead, cfg.df_lookahead) + (cfg.df_lookahead if kind == "dfn2" else 0)
    outs, pos = [], 0
    for i, k in enumerate([1, 1, 2, 1, 7, 40, 1, 3, 64, 30, 7]):
        x = audio[:, pos * hop:(pos + k) * hop]
        outs.append(s.process(x.cuda() if i % 2 else x).cpu())
        pos += k
    assert pos == n
    outs.append(s.flush())
    got = torch.cat(outs, 1)
    lat = s.latency_frames * hop
    assert got.shape == (2, n * hop + lat)
    assert lat == 0 or got[:, :lat].abs().max() == 0
    assert rms(got[:, lat:], ref) < 1e-6
    # a reset stream reproduces itself; atten_lim is honoured
    s.reset()
    again = torch.cat([s.process(audio), s.flush()], 1)
    assert rms(again, got) < 1e-6
    s2 = DfStream(model, st, batch=2, atten_lim_db=12.0)
    lim = torch.cat([s2.process(audio), s2.flush()], 1)[:, lat:]
    assert rms(lim, enhance(model, st, audio, pad=False, atten_lim_db=12.0)) < 1e-6


# ------------------------------------------------------------------ callers either side of the path (SURVEY 8f-3, 8f-4) ----
@pytest.mark.parametrize("orig,new,method", [(44100, 48000, "sinc_fast"), (48000, 16000, "sinc_best"), (16000, 48000, "kaiser_fast"),
                                             (48000, 44100, "kaiser_best")])
def test_resample_matches_torchaudio(orig, new, method):
    """df.io.resample (io.py:107-129): the CUDA polyphase kernel against torchaudio.functional.resample -- the reference's
    own dependency for this step -- with the reference's parameter sets."""
    ta = pytest.importorskip("torchaudio")
    from deepfilternet_b200.io import get_resample_params, resample
    x = synth_audio(2, orig // 2 + 17, seed=3, sr=orig)
    got = resample(x, orig, new, method=method)
    ref = ta.functional.resample(x, orig, new, **get_resample_params(method))
    assert got.shape == ref.shape and float((got - ref).abs().max()) < 2e-6
    assert resample(x, orig, orig) is x


def test_audio_io_and_cli_roundtrip(tmp_path, golden_dir, model_dir):
    """df.io load_audio / save_audio on WAV files and the `deepFilter` CLI (enhance.py:47-89, 299-379): the file the CLI
    writes equals enhance() of the loaded audio, int16-scaled like io.py:80-85."""
    import ref_harness as rh
    from deepfilternet_b200 import io as dio
    from deepfilternet_b200.enhance import run
    src = os.path.join(golden_dir, "assets", "noisy_snr0.wav")
    audio, meta = dio.load_audio(src, 48000)
    assert meta.sample_rate == 48000 and audio.shape[0] == meta.num_channels == 1
    assert np.array_equal(audio.numpy(), rh.read_wav(src))
    out_dir = tmp_path / "out"
    assert run(["-m", os.path.join(model_dir, "DeepFilterNet3"), "-o", str(out_dir), "--log-level", "ERROR", src]) == 0
    written, wmeta = dio.load_audio(str(out_dir / "noisy_snr0_DeepFilterNet3.wav"))
    model, st, _, _ = init_df(os.path.join(model_dir, "DeepFilterNet3"), log_level="ERROR")
    ref = (enhance(model, st, audio) * (1 << 15)).to(torch.int16).to(torch.float32) / 32768.0
    assert wmeta.sample_rate == 48000 and written.shape == ref.shape
    assert float((written - ref).abs().max()) <= 1.0 / 32768.0 + 1e-7
    # float32 files and a rate the model does not run at: resampled in, resampled back out
    x16 = dio.resample(audio[:, :48000], 48000, 16000)
    p16 = dio.save_audio(str(tmp_path / "a16.wav"), x16, 16000, dtype=torch.float32)
    back, m16 = dio.load_audio(p16, 48000, verbose=False)
    assert m16.sample_rate == 16000 and m16.encoding == "PCM_F" and back.shape[1] == 48000


def test_training_feature_producer(states):
    """SURVEY 8(f)-4: FftDataset::get_sample's transform (dataset.rs:863-914) on device tensors == the oracle's
    analysis -> erb -> erb_norm / unit_norm."""
    from deepfilternet_b200.features import fft_features
    st, ost = states
    noisy, speech = synth_audio(3, 24000, seed=5), synth_audio(3, 24000, seed=6)
    out = fft_features(st, noisy.cuda(), speech.cuda(), nb_spec=96, norm_alpha=0.99)
    spec = ost.analysis(noisy.numpy())
    assert np.abs(out["noisy"].cpu().numpy()[:, 0] - np.stack([spec.real, spec.imag], -1)).max() < 1e-6
    sp = ost.analysis(speech.numpy())
    assert np.abs(out["speech"].cpu().numpy()[:, 0] - np.stack([sp.real, sp.imag], -1)).max() < 1e-6
    assert np.abs(out["feat_erb"].cpu().numpy()[:, 0] - LO.erb_norm(LO.erb(spec, ost.erb_widths()), 0.99)).max() < 2e-6
    un = LO.unit_norm(np.ascontiguousarray(spec[..., :96]), 0.99)
    assert np.abs(out["feat_spec"].cpu().numpy()[:, 0] - np.stack([un.real, un.imag], -1)).max() < 1e-5


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_post_filter_and_mask_only(name, golden_dir, model_dir):
    """init_df(post_filter=True) / init_df(mask_only=True) against the reference modules' outputs
    (tests/golden/dfnet_pf.npz, oracle/gen_golden_pf.py) and, in streaming mode, against the one-shot path."""
    from deepfilternet_b200 import DfStream
    g = np.load(os.path.join(golden_dir, "dfnet_pf.npz"))
    audio = torch.from_numpy(g["audio"])
    model, st, suffix, _ = init_df(os.path.join(model_dir, name), post_filter=True, log_level="ERROR")
    assert suffix == name + "_pf" and model.post_filter
    assert rms(enhance(model, st, audio), g[f"{name}_pf"]) < RMS_TOL
    assert rms(enhance(model, st, audio, atten_lim_db=12.0), g[f"{name}_pf_atten12"]) < RMS_TOL
    x = audio[:, :480 * 50]
    s = DfStream(model, st, batch=2)
    got = torch.cat([s.process(x[:, :480 * 7]), s.process(x[:, 480 * 7:]), s.flush()], 1)[:, s.latency_frames * 480:]
    assert rms(got, enhance(model, st, x, pad=False)) < 1e-6
    model, st, _, _ = init_df(os.path.join(model_dir, name), mask_only=True, log_level="ERROR")
    assert not model.run_df
    assert rms(enhance(model, st, audio), g[f"{name}_mask_only"]) < RMS_TOL


def test_streaming_lsnr_stage_gating(states):
    """tract.rs:658-672 `apply_stages` on the streaming path: thresholds that force one stage for every frame must
    reproduce that stage's definition -- gains + DF (the ungated output), gains only (== mask_only), unprocessed (== the
    noisy input through STFT/ISTFT), zero gains (silence) -- and the atten limit mixes the noisy signal back in."""
    from deepfilternet_b200 import DfStream
    st, _ = states
    cfg = cfg_of("dfn3")
    sd = random_state_dict(cfg, seed=15)
    model = DfNet(cfg, sd, st)
    hop, n = 480, 90
    audio = synth_audio(2, hop * n, seed=81)

    def run(model, **th):
        s = DfStream(model, st, batch=2, atten_lim_db=th.pop("atten", None))
        if th:
            s.set_lsnr_thresholds(**th)
        return torch.cat([s.process(audio[:, :hop * 33]), s.process(audio[:, hop * 33:]), s.flush()], 1)[:, s.latency_frames * hop:]

    base = run(model)
    assert rms(run(model, min_db_thresh=-1e9, max_db_erb_thresh=1e9, max_db_df_thresh=1e9), base) < 1e-7      # always stage 3
    gains_only = run(model, min_db_thresh=-1e9, max_db_erb_thresh=1e9, max_db_df_thresh=-1e9)                 # always stage 2
    mo = DfNet(cfg, sd, st, run_df=False)
    assert rms(gains_only, run(mo)) < 1e-7 and rms(gains_only, base) > 1e-5
    passthrough = run(model, min_db_thresh=-1e9, max_db_erb_thresh=-1e9, max_db_df_thresh=-1e9)               # always stage 1
    ident = torch.from_numpy(st.synthesis(st.analysis(audio.numpy())))
    assert rms(passthrough, ident) < 1e-6
    assert run(model, min_db_thresh=1e9, max_db_erb_thresh=2e9, max_db_df_thresh=2e9).abs().max() < 1e-7      # always stage 0
    lim = 10 ** (-12 / 20)
    z = run(model, min_db_thresh=1e9, max_db_erb_thresh=2e9, max_db_df_thresh=2e9, atten=12.0)
    assert rms(z, ident * lim) < 1e-6


# ------------------------------------------------------------------ DeepFilterNet v1 (SURVEY.md 8f-2) ----
def cfg_v1():
    return ModelConfig(model="deepfilternet", conv_lookahead=2, df_lookahead=1, conv_ch=64, conv_kernel=(2, 3), convt_kernel=(2, 3),
                       conv_kernel_inp=(2, 3), conv_k_enc=2, conv_k_dec=2, emb_hidden_dim=512, df_hidden_dim=512, emb_num_layers=3,
                       df_num_layers=2, gru_groups=8, lin_groups=8, enc_lin_groups=8, group_shuffle=True, dfop_method="real_unfold")


def test_v1_golden_reference_outputs(golden_dir, model_dir):
    """DeepFilterNet (v1: convkxf with in-conv look-ahead, GroupedGRU / GroupedLinear with shuffle, DfOp with alpha) against
    outputs of the reference's own modules (tests/golden/dfnet_DeepFilterNet.npz, made by oracle/gen_golden_v1.py)."""
    g = np.load(os.path.join(golden_dir, "dfnet_DeepFilterNet.npz"))
    model, st, suffix, epoch = init_df(os.path.join(model_dir, "DeepFilterNet"), log_level="ERROR")
    assert suffix == "DeepFilterNet" and epoch == int(g["epoch"]) and model.cfg.model == "deepfilternet"
    spec_e, m, lsnr, alpha = model(torch.from_numpy(g["spec"]), torch.from_numpy(g["feat_erb"]), torch.from_numpy(g["feat_spec"]))
    assert rms(m, g["m"]) < TOL_M and np.abs(lsnr.numpy() - g["lsnr"]).max() < TOL_LSNR
    assert alpha.shape == g["alpha"].shape and np.abs(alpha.numpy() - g["alpha"]).max() < 1e-4
    assert rms(spec_e, g["spec_e"]) < TOL_SPEC
    audio = torch.from_numpy(g["audio"])
    assert rms(enhance(model, st, audio), g["enhanced"]) < RMS_TOL
    o = enhance(model, st, audio, pad=False)
    assert o.shape == g["enhanced_nopad"].shape and rms(o, g["enhanced_nopad"]) < RMS_TOL
    assert rms(enhance(model, st, audio, atten_lim_db=12.0), g["enhanced_atten12"]) < RMS_TOL
    assert rms(enhance(model, st, torch.from_numpy(g["audio2"])), g["enhanced2"]) < RMS_TOL
    with pytest.raises(_lib.DfbError, match="one window per signal"):   # no frame-incremental API for v1
        from deepfilternet_b200 import DfStream
        DfStream(model, st, 1)


def test_v1_si_sdr_known_answer_and_whole_asset(golden_dir, model_dir):
    """The third known answer check of the reference CI (df/scripts/test_df.py:45-55: DeepFilterNet) on the CUDA path, and
    every sample of the 10.6 s recording against the oracle."""
    import dfnet1_oracle as O1
    import ref_harness as rh
    kat = json.load(open(os.path.join(golden_dir, "kat.json")))["DeepFilterNet"]
    model, st, _, epoch = init_df(os.path.join(model_dir, "DeepFilterNet"), log_level="ERROR")
    assert epoch == kat["epoch"]
    noisy = torch.from_numpy(rh.read_wav(os.path.join(golden_dir, "assets", "noisy_snr0.wav")))
    clean = rh.read_wav(os.path.join(golden_dir, "assets", "clean_freesound_33711.wav"))
    out = enhance(model, st, noisy, pad=True)
    s = rh.si_sdr(clean, out.numpy())
    assert abs(s - kat["target"]) <= 1e-4 + 1e-4 * abs(kat["target"]), (s, kat["target"])
    ref = O1.enhance(model.state_dict(), dict(O1.DEFAULTS_DFN1), noisy)
    assert out.shape == ref.shape and rms(out, ref) < RMS_TOL


@pytest.mark.parametrize("precision", ["fp32+gru_tc+proj_tc+conv_tc", "fp32"])
@pytest.mark.parametrize("B,T", [(3, 24000), (1, 4800), (9, 9600 + 123)])
def test_v1_random_weights_vs_oracle(states, B, T, precision):
    """Random weights (BatchNorm statistics included) so that the packing -- folded shuffles, gather tables, block-diagonal
    GRUs, reversed transposed-conv taps -- is exercised away from the trained checkpoint; both arithmetic modes."""
    import dfnet1_oracle as O1
    st, _ = states
    cfg = cfg_v1()
    sd = random_state_dict(cfg, seed=7)
    model = DfNet(cfg, sd, st)
    model.set_precision(precision)
    audio = synth_audio(B, T, seed=23)
    out_o, aux = O1.enhance(sd, dict(O1.DEFAULTS_DFN1), audio, return_all=True)
    spec_e, m, lsnr, alpha = model(aux["spec"], aux["erb_feat"], aux["spec_feat"])
    assert rms(m, aux["m"]) < TOL_M and rms(spec_e, aux["spec_e"]) < TOL_SPEC
    assert np.abs(lsnr.numpy() - aux["lsnr"].numpy()).max() < TOL_LSNR and np.abs(alpha.numpy() - aux["alpha"].numpy()).max() < 1e-4
    out = enhance(model, st, audio)
    assert out.shape == audio.shape and rms(out, out_o) < RMS_TOL
    dev = enhance_device(model, st, audio.cuda())
    assert rms(dev.cpu(), out_o) < RMS_TOL


def test_v1_stream_groups_and_independence(states):
    """Stream groups under a small workspace cap (one window per signal, so only the batch is split) and batch-position
    independence."""
    import dfnet1_oracle as O1
    st, _ = states
    cfg = cfg_v1()
    sd = random_state_dict(cfg, seed=8)
    model = DfNet(cfg, sd, st)
    audio = synth_audio(11, 24000, seed=29).cuda()
    full = enhance_device(model, st, audio)
    model.set_max_workspace(48 << 20)   # a few streams per group
    grouped = enhance_device(model, st, audio)
    model.set_max_workspace(64 << 30)
    assert rms(full.cpu(), grouped.cpu()) < 1e-7
    assert rms(full[4:5].cpu(), O1.enhance(sd, dict(O1.DEFAULTS_DFN1), audio[4:5].cpu())) < RMS_TOL
    single = enhance_device(model, st, audio[10:11].contiguous())
    assert rms(full[10:11].cpu(), single.cpu()) < 1e-7
