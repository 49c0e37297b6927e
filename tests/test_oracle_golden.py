"""CPU: the oracle (oracle/) against every golden vector / known answer the reference's own tests
hold for this path (SURVEY.md 8c)."""
import json
import os

import numpy as np
import pytest
import torch

import dfnet_oracle as O
import libdf_oracle as LO

from deepfilternet_b200.config import load_config
from deepfilternet_b200.model import find_checkpoint, load_state_dict_file


def test_erb_widths_match_checkpoint_buffers(golden_dir):
    """libDF/src/lib.rs:68-100 must reproduce the band layout stored in the shipped `erb_fb` buffers."""
    g = json.load(open(os.path.join(golden_dir, "erb_widths.json")))
    p = g["params"]
    w = LO.erb_widths(p["sr"], p["fft_size"], p["nb_bands"], p["min_nb_freqs"])
    for name, ref in g["from_checkpoint_erb_fb"].items():
        assert w.tolist() == ref, name
    assert int(w.sum()) == p["fft_size"] // 2 + 1


def test_stft_istft_delay():
    """libDF/src/transforms.rs:618-638 (test_stft_istft_delay): correlation > 1 - 1e-6 after the
    n_fft - hop delay."""
    rng = np.random.default_rng(0)
    st = LO.DF(48000, 960, 480, 32, 2)
    x = (rng.standard_normal((1, 48000)) * 0.1).astype(np.float32)
    y = st.synthesis(st.analysis(x))
    d = 960 - 480
    a, b = x[0, : -d], y[0, d:]
    corr = float(np.dot(a, b) / np.sqrt(np.dot(a, a) * np.dot(b, b)))
    assert corr > 1 - 1e-6
    assert np.abs(a - b).max() < 1e-5


def test_band_gain_exact():
    """libDF/src/lib.rs:626-652 (test_erb_inout): band gains multiply every bin of the band exactly."""
    w = LO.erb_widths(24000, 192, 24, 1)
    rng = np.random.default_rng(1)
    x = (rng.uniform(-1, 1, (1, 97)) + 1j * rng.uniform(-1, 1, (1, 97))).astype(np.complex64)
    mask = np.ones((1, 24), dtype=np.float32)
    mask[0, 3], mask[0, 23] = 0.3, 0.5
    gains = LO.erb_inv(mask, w)
    out = x * gains
    o = 0
    for b, n in enumerate(w):
        assert np.array_equal(out[0, o:o + n], x[0, o:o + n] * mask[0, b])
        o += n


def test_erb_identity():
    """DeepFilterNet/df/modules.py:929-947 (test_erb): libdf.erb(db=False) == |X|^2 @ erb_fb."""
    rng = np.random.default_rng(2)
    w = LO.erb_widths(48000, 960, 32, 2)
    x = (rng.standard_normal((2, 5, 481)) + 1j * rng.standard_normal((2, 5, 481))).astype(np.complex64)
    fb = np.zeros((481, 32), dtype=np.float32)
    o = 0
    for b, n in enumerate(w):
        fb[o:o + n, b] = 1.0 / n
        o += n
    ref = (np.abs(x) ** 2) @ fb
    assert np.allclose(LO.erb(x, w, db=False), ref, rtol=1e-5, atol=1e-6)


def test_unit_norm_matches_exponential_unit_norm():
    """modules.py:950-967 (test_unit_norm): libdf.unit_norm == ExponentialUnitNorm recursion."""
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((1, 20, 96)) + 1j * rng.standard_normal((1, 20, 96))).astype(np.complex64)
    a = 0.99
    out = LO.unit_norm(x, a)
    s = LO.unit_norm_init(96)[0].astype(np.float32)
    for t in range(20):
        s = np.abs(x[0, t]).astype(np.float32) * np.float32(1 - a) + s * np.float32(a)
        assert np.allclose(out[0, t], x[0, t] / np.sqrt(s), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_dfnet_oracle_matches_reference_modules(name, golden_dir, model_dir):
    """tests/golden/dfnet_<model>.npz were produced by the reference's own DfNet / enhance() with the same weights."""
    g = np.load(os.path.join(golden_dir, f"dfnet_{name}.npz"))
    cfg = load_config(os.path.join(model_dir, name, "config.ini"), env={})
    sd = load_state_dict_file(find_checkpoint(os.path.join(model_dir, name, "checkpoints"))[0])
    audio = torch.from_numpy(g["audio"])
    out, aux = O.enhance(sd, cfg.as_dict(), audio, pad=True, return_all=True)
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


def test_ll_oracle_matches_reference_modules(golden_dir, model_dir):
    """tests/golden/dfnet_DeepFilterNet3_ll.npz holds the outputs of the reference DfNet built from the _ll config
    (H = 512, zero look-ahead, kt = 2 convs)."""
    d = os.path.join(model_dir, "DeepFilterNet3_ll")
    cfg = load_config(os.path.join(d, "config.ini"), env={})
    sd = load_state_dict_file(find_checkpoint(os.path.join(d, "checkpoints"))[0])
    g = np.load(os.path.join(golden_dir, "dfnet_DeepFilterNet3_ll.npz"))
    out, aux = O.enhance(sd, cfg.as_dict(), torch.from_numpy(g["audio"]), pad=True, return_all=True)
    assert np.abs(aux["m"].numpy() - g["m"]).max() < 1e-5
    assert np.abs(aux["spec_e"].numpy() - g["spec_e"]).max() < 1e-6
    assert float(np.sqrt(((out.numpy() - g["enhanced"]) ** 2).mean())) < 1e-6


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_si_sdr_known_answer(name, golden_dir, model_dir):
    """DeepFilterNet/df/scripts/test_df.py:44-78 on the weights of model_dir: SI-SDR of enhance(noisy_snr0) vs clean against
    the reference modules' value (tests/golden/kat.json), atol=rtol=1e-4."""
    import ref_harness as rh
    kat = json.load(open(os.path.join(golden_dir, "kat.json")))[name]
    cfg = load_config(os.path.join(model_dir, name, "config.ini"), env={})
    sd = load_state_dict_file(find_checkpoint(os.path.join(model_dir, name, "checkpoints"))[0])
    noisy = torch.from_numpy(rh.read_wav(os.path.join(golden_dir, "assets", "noisy_snr0.wav")))
    clean = rh.read_wav(os.path.join(golden_dir, "assets", "clean_freesound_33711.wav"))
    assert noisy.shape[1] == kat["n_samples"]
    out = O.enhance(sd, cfg.as_dict(), noisy, pad=True)
    s = rh.si_sdr(clean, out.numpy())
    assert abs(s - kat["target"]) <= 1e-4 + 1e-4 * abs(kat["target"]), (s, kat["target"])


def test_oracle_carried_state_semantics():
    """pyDF `reset` argument (pyDF/src/lib.rs:56-58, 91-93; DFState::reset libDF/src/lib.rs:156-159) in the oracle that
    the GPU `libdf` mirror is checked against: chunked `reset=False` streaming of one channel equals the one-shot
    transform, channel c continues channel c - 1, and a `reset=True` call clears BOTH memories first."""
    import libdf_oracle as LO
    from tests_common import synth_audio
    st = LO.DF(48000, 960, 480, 32, 2)
    x = synth_audio(2, 9600, seed=8).numpy()
    whole = st.analysis(x[:1], reset=True)
    st.reset()
    parts = np.concatenate([st.analysis(np.ascontiguousarray(x[:1, o:o + 2400]), reset=False) for o in range(0, 9600, 2400)], 1)
    assert np.array_equal(whole, parts)
    # two channels without reset == the concatenated signal in one channel
    st.reset()
    two = st.analysis(x, reset=False)
    st.reset()
    cat = st.analysis(x.reshape(1, -1), reset=True)
    assert np.array_equal(two.reshape(1, -1, 481), cat)
    # synthesis: chunked streaming == one shot; and analysis(reset=True) wipes the synthesis memory as well
    st.reset()
    y_whole = st.synthesis(whole.copy(), reset=True)
    st.reset()
    y_parts = np.concatenate([st.synthesis(whole[:, o:o + 5].copy(), reset=False) for o in range(0, 20, 5)], 1)
    assert np.array_equal(y_whole, y_parts)
    st.synthesis(whole.copy(), reset=True)       # leaves a non-zero synthesis memory behind
    st.analysis(x[:1], reset=True)               # DFState::reset clears it
    assert np.array_equal(st.synthesis(whole.copy(), reset=False), y_whole)


@pytest.mark.parametrize("name", ["DeepFilterNet3", "DeepFilterNet2"])
def test_oracle_post_filter_and_mask_only_match_reference_modules(name, golden_dir, model_dir):
    """The optional stages: `init_df(post_filter=True)` (deepfilternet3.py:448-454 on the spectrum; DFN2: Mask.pf on the
    ERB gains, modules.py:234-245) and `mask_only=True` (run_df = False), pinned to the reference modules' outputs
    (tests/golden/dfnet_pf.npz, made by oracle/gen_golden_pf.py)."""
    g = np.load(os.path.join(golden_dir, "dfnet_pf.npz"))
    d = os.path.join(model_dir, name)
    cfg = load_config(os.path.join(d, "config.ini"), env={})
    sd = load_state_dict_file(find_checkpoint(os.path.join(d, "checkpoints"))[0])
    audio = torch.from_numpy(g["audio"])
    rmsd = lambda a, b: float(np.sqrt(((a.numpy() - b) ** 2).mean()))
    c = dict(cfg.as_dict(), mask_pf=True)
    assert rmsd(O.enhance(sd, c, audio), g[f"{name}_pf"]) < 1e-6
    assert rmsd(O.enhance(sd, c, audio, atten_lim_db=12.0), g[f"{name}_pf_atten12"]) < 1e-6
    c = dict(cfg.as_dict(), mask_only=True)
    assert rmsd(O.enhance(sd, c, audio), g[f"{name}_mask_only"]) < 1e-6
    # and they are not no-ops
    assert rmsd(O.enhance(sd, cfg.as_dict(), audio), g[f"{name}_pf"]) > 1e-5


def test_v1_oracle_matches_reference_modules(golden_dir, model_dir):
    """oracle/dfnet1_oracle.py against outputs of the reference's own DeepFilterNet (v1) modules (oracle/gen_golden_v1.py)."""
    import dfnet1_oracle as O1
    g = np.load(os.path.join(golden_dir, "dfnet_DeepFilterNet.npz"))
    cfg = load_config(os.path.join(model_dir, "DeepFilterNet", "config.ini"), env={})
    assert (cfg.model, cfg.gru_groups, cfg.lin_groups, cfg.conv_k_enc, cfg.conv_k_dec, cfg.df_lookahead) == ("deepfilternet", 8, 8, 2, 2, 1)
    path, epoch = find_checkpoint(os.path.join(model_dir, "DeepFilterNet", "checkpoints"))
    assert epoch == int(g["epoch"])
    sd = load_state_dict_file(path)
    ocfg = dict(O1.DEFAULTS_DFN1)
    for k in ("conv_lookahead", "df_lookahead", "df_order", "nb_df", "nb_erb", "emb_num_layers", "df_num_layers", "gru_groups", "lin_groups",
              "conv_k_enc", "conv_k_dec", "group_shuffle"):
        assert ocfg[k] == getattr(cfg, k), k
    st = LO.DF(48000, 960, 480, 32, 2)
    spec_e, m, lsnr, coefs, alpha = O1.dfnet1_forward(sd, ocfg, st.erb_widths(), torch.from_numpy(g["spec"]), torch.from_numpy(g["feat_erb"]),
                                                      torch.from_numpy(g["feat_spec"]))
    assert np.abs(spec_e.numpy() - g["spec_e"]).max() < 1e-6 and np.abs(m.numpy() - g["m"]).max() < 5e-6
    assert np.abs(lsnr.numpy() - g["lsnr"]).max() < 1e-4 and np.abs(alpha.numpy() - g["alpha"]).max() < 5e-6
    audio = torch.from_numpy(g["audio"])
    assert np.abs(O1.enhance(sd, ocfg, audio).numpy() - g["enhanced"]).max() < 1e-6
    assert np.abs(O1.enhance(sd, ocfg, audio, pad=False).numpy() - g["enhanced_nopad"]).max() < 1e-6
    assert np.abs(O1.enhance(sd, ocfg, audio, atten_lim_db=12.0).numpy() - g["enhanced_atten12"]).max() < 1e-6
    assert np.abs(O1.enhance(sd, ocfg, torch.from_numpy(g["audio2"])).numpy() - g["enhanced2"]).max() < 1e-6


def test_v1_si_sdr_known_answer(golden_dir, model_dir):
    """df/scripts/test_df.py:45-55 for DeepFilterNet (v1) on the weights of model_dir, atol = rtol = 1e-4."""
    import dfnet1_oracle as O1
    import ref_harness as rh
    kat = json.load(open(os.path.join(golden_dir, "kat.json")))["DeepFilterNet"]
    sd = load_state_dict_file(find_checkpoint(os.path.join(model_dir, "DeepFilterNet", "checkpoints"))[0])
    noisy = torch.from_numpy(rh.read_wav(os.path.join(golden_dir, "assets", "noisy_snr0.wav")))
    clean = rh.read_wav(os.path.join(golden_dir, "assets", "clean_freesound_33711.wav"))
    out = O1.enhance(sd, dict(O1.DEFAULTS_DFN1), noisy, pad=True)
    s = rh.si_sdr(clean, out.numpy())
    assert abs(s - kat["target"]) <= 1e-4 + 1e-4 * abs(kat["target"]), (s, kat["target"])
