"""The oracle held to outputs of the REFERENCE'S OWN CODE.

tests/golden/ref_executed_models.npz is written by scripts/make_golden_ref.py, which imports the reference's model files from
a checkout of it and runs them - FastSpeech2.inference / forward / FastSpeech2Loss, PWGGenerator.forward (plain and through the
reference's own apply_weight_norm), ConditionalWaveFlow encoder + WaveFlow.inverse - on a torch-backed stand-in for the Paddle
primitives they call (scripts/refexec/paddle_standin.py), with the oracle's seeded Paddle-layout state dicts loaded into the
reference classes.  That run also asserts that every state-dict key and shape of the reference's class tree equals ours.
The vectors travel with the repo (large arrays as samples, tests/golden_sample.py); these tests need neither the reference
nor a GPU."""
import os

import numpy as np
import pytest
import torch

import golden_sample as gs
from conftest import rel_err

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = 2e-6        # same arithmetic, same torch kernels underneath: the oracle reproduces the executed reference to rounding


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLD, "ref_executed_models.npz"))


def test_state_dict_keys_equal_the_reference_class_trees(g):
    from oracle import fastspeech2 as ofs
    from oracle import pwg as opwg
    from oracle import waveflow as owf
    assert sorted(ofs.synth_params(1)) == list(g["fs2_keys"])
    assert sorted(opwg.fold_weight_norm(opwg.synth_params(2, weight_norm=True))) == list(g["pwg_keys"])
    assert sorted(opwg.synth_params(2, weight_norm=True)) == list(g["pwg_wn_keys"])
    assert sorted(owf.synth_params(4)) == list(g["wf_keys"])
    # and the CUDA-side host classes expose exactly the same names (the checkpoint boundary of SURVEY 8b)
    from parakeet_b200.models import ConditionalWaveFlow, FastSpeech2, PWGGenerator
    fs = FastSpeech2(80, 80, **ofs.LJSPEECH_MODEL_CFG, device="cpu")
    assert sorted(fs.state_dict()) == list(g["fs2_keys"])
    gen = PWGGenerator(**opwg.DEFAULT_GENERATOR_PARAMS, device="cpu")
    assert sorted(gen.state_dict()) == list(g["pwg_wn_keys"])
    wf = ConditionalWaveFlow([16, 16], 8, 8, 16, 64, 80, (3, 3), device="cpu")
    assert sorted(wf.state_dict()) == list(g["wf_keys"])


def test_fastspeech2_oracle_equals_executed_reference(g):
    from oracle import fastspeech2 as ofs
    params = ofs.synth_params(1)
    text = torch.from_numpy(g["fs2_inf_text"])
    with torch.no_grad():
        mel = ofs.fs2_inference(params, None, text)
        mel13 = ofs.fs2_inference(params, None, text, alpha=1.3)
    assert tuple(mel.shape) == gs.shape(g, "fs2_inf_mel") and gs.err(mel, g, "fs2_inf_mel") < TOL
    assert tuple(mel13.shape) == gs.shape(g, "fs2_inf_mel_alpha") and gs.err(mel13, g, "fs2_inf_mel_alpha") < TOL
    b = gs.fs2_batch(g, "fs2_fwd")
    with torch.no_grad():
        out = ofs.fs2_forward(params, None, b["text"], b["text_lengths"], b["speech_lengths"], b["durations"], b["pitch"], b["energy"])
    for name, t in zip(("before", "after", "d_outs", "p_outs", "e_outs"), out[:5]):
        assert tuple(t.shape) == gs.shape(g, f"fs2_fwd_out_{name}") and gs.err(t, g, f"fs2_fwd_out_{name}") < TOL, name
    before, after, d_outs, p_outs, e_outs = out[:5]
    losses = ofs.fs2_loss(after, before, d_outs, p_outs, e_outs, b["speech"], b["durations"], b["pitch"], b["energy"], b["text_lengths"],
                          b["speech_lengths"])
    assert np.allclose([float(v) for v in losses[:4]], g["fs2_loss"], rtol=1e-5)       # l1, duration, pitch, energy


def test_pwg_oracle_equals_executed_reference(g):
    from oracle import pwg as opwg
    wn = opwg.synth_params(2, weight_norm=True)
    x, c = torch.from_numpy(g["pwg_x"]), torch.from_numpy(g["pwg_c"])
    with torch.no_grad():
        y = opwg.generator_forward(opwg.fold_weight_norm(wn), x, c)
    assert gs.err(y, g, "pwg_y") < TOL
    assert gs.err(y, g, "pwg_y_weight_norm") < 1e-5                                  # the reference's own weight_norm(g, v) path


def test_waveflow_oracle_equals_executed_reference(g):
    from oracle import waveflow as owf
    folded = owf.fold_weight_norm(owf.synth_params(4))
    mel, z = torch.from_numpy(g["wf_mel"]), torch.from_numpy(g["wf_z"])
    with torch.no_grad():
        cond = owf.encoder(folded, mel, 2)
        x = owf.infer(folded, mel, z)
    assert gs.err(cond, g, "wf_cond") < 1e-5
    assert tuple(x.shape) == gs.shape(g, "wf_x") and gs.err(x, g, "wf_x") < 1e-5
    # 22 mel frames: W = 335 > 2 x 128, the widest (+-128) width taps of layer 7 read live columns in the reference
    mel2, z2 = torch.from_numpy(g["wf2_mel"]), torch.from_numpy(g["wf2_z"])
    assert z2.shape[-1] // 16 > 2 * 128
    with torch.no_grad():
        x2 = owf.infer(folded, mel2, z2)
    assert tuple(x2.shape) == gs.shape(g, "wf2_x") and gs.err(x2, g, "wf2_x") < 1e-5
    # the shipped config (examples/waveflow/config.py: 128 residual channels), W = 335
    folded128 = owf.fold_weight_norm(owf.synth_params(5, channels=128))
    mel3, z3 = torch.from_numpy(g["wf128_mel"]), torch.from_numpy(g["wf128_z"])
    with torch.no_grad():
        x3 = owf.infer(folded128, mel3, z3)
    assert tuple(x3.shape) == gs.shape(g, "wf128_x") and gs.err(x3, g, "wf128_x") < 1e-5


def test_inference_wrappers_and_stft_equal_executed_reference(g):
    """FastSpeech2Inference (inference + ZScore.inverse), PWGInference (ZScore + replicate padding + transposes, the reference's
    own inference() with the noise supplied) and modules/audio.STFT (DFT-matrix conv, real / imag / magnitude)."""
    from oracle import fastspeech2 as ofs
    from oracle import pwg as opwg
    from oracle import stft as ostft
    mu, sigma = torch.from_numpy(g["wr_mu"]), torch.from_numpy(g["wr_sigma"])
    with torch.no_grad():
        logmel = ofs.fs2_inference_denorm(ofs.synth_params(1), None, torch.from_numpy(g["wr_text"]), mu, sigma)
    assert tuple(logmel.shape) == gs.shape(g, "wr_logmel") and gs.err(logmel, g, "wr_logmel") < TOL
    folded = opwg.fold_weight_norm(opwg.synth_params(2, weight_norm=True))
    with torch.no_grad():
        wav = opwg.pwg_inference(folded, torch.from_numpy(g["wr_pwg_logmel"]), mu, sigma, torch.from_numpy(g["wr_pwg_noise"]))
    assert tuple(wav.shape) == gs.shape(g, "wr_pwg_wav") and gs.err(wav, g, "wr_pwg_wav") < TOL
    x = torch.from_numpy(g["stft_x"])
    for tag, (n_fft, hop, win) in (("a", (512, 128, 512)), ("b", (1024, 120, 600))):
        re, im = ostft.stft_dft_conv(x, n_fft, hop, win)
        assert gs.err(re, g, f"stft_{tag}_re") < 1e-5 and gs.err(im, g, f"stft_{tag}_im") < 1e-5
        assert gs.err(torch.sqrt(re ** 2 + im ** 2), g, f"stft_{tag}_mag") < 1e-5


def test_multi_resolution_stft_loss_equals_executed_reference(g):
    from oracle import stft as ostft
    sc, mag = ostft.multi_resolution_stft_loss(torch.from_numpy(g["stft_x"]), torch.from_numpy(g["mrstft_y"]))
    assert np.allclose([float(sc), float(mag)], g["mrstft_loss"], rtol=2e-5)


def test_training_forward_loss_and_gradients_equal_executed_reference(g):
    """The reference model in train mode (dropout 0, BatchNorm on batch statistics) + its FastSpeech2Loss + the updater's loss sum,
    differentiated by autograd THROUGH THE REFERENCE'S CODE: losses, a representative set of gradients (every kind of tensor on
    the path, large ones sampled, + their norms) and the updated BatchNorm statistics vs oracle.train_step_grads - the reference
    the CUDA training step is tested against."""
    from oracle import fastspeech2 as ofs
    params = ofs.synth_params(1)
    b = gs.fs2_batch(g, "fs2_train")
    losses, grads, stats = ofs.train_step_grads(params, None, b)
    assert np.allclose([losses["l1_loss"], losses["duration_loss"], losses["pitch_loss"], losses["energy_loss"]], g["fs2_train_loss"], rtol=1e-5)
    keys = [k[len("fs2_train_grad/"):] for k in g.files if k.startswith("fs2_train_grad/")]
    assert len(keys) == 18
    for k in keys:
        assert gs.err(grads[k], g, "fs2_train_grad/" + k) < 2e-4, k     # fp32 autograd through two orderings of the same graph
        assert abs(float(grads[k].double().norm()) - float(g["fs2_train_gradnorm/" + k])) <= 2e-4 * max(float(g["fs2_train_gradnorm/" + k]), 1e-12), k
    for k in [k for k in g.files if k.startswith("fs2_train_stat/")]:
        assert rel_err(stats[k[len("fs2_train_stat/"):]], torch.from_numpy(g[k])) < 1e-5, k


def test_pwg_discriminator_equals_executed_reference(g):
    from oracle import pwg as opwg
    dp = opwg.synth_discriminator_params(12)
    assert sorted(dp) == list(g["pwgd_keys"])
    with torch.no_grad():
        y = opwg.discriminator_forward(dp, torch.from_numpy(g["pwgd_x"]))
    assert gs.err(y, g, "pwgd_y") < TOL


def test_multispeaker_tone_oracle_equals_executed_reference(g):
    """aishell3 / vctk shape (speaker table + projection, concat or add) with tone embeddings: the reference's own
    inference(spk_id, tone_id) and batched forward(..., tone_id, spk_id) against the oracle, both integration types."""
    from oracle import fastspeech2 as ofs
    for tag, (st, tt) in (("a", ("concat", "add")), ("b", ("add", "concat"))):
        p = ofs.add_speaker_tone_params(ofs.synth_params(1), 1, spk_type=st, tone_type=tt)
        assert sorted(p) == list(g[f"fs2ms_{tag}_keys"])
        cfg = dict(spk_embed_integration_type=st, tone_embed_integration_type=tt)
        text, tone = torch.from_numpy(g[f"fs2ms_{tag}_inf_text"]), torch.from_numpy(g[f"fs2ms_{tag}_inf_tone"])
        with torch.no_grad():
            out = ofs.fs2_forward(p, cfg, text.unsqueeze(0), torch.tensor([text.shape[0]]), is_inference=True, spk_id=torch.tensor([4]),
                                  tone_id=tone.unsqueeze(0) if tt == "add" else None, tone_per_utterance=True)
        assert tuple(out[1][0].shape) == gs.shape(g, f"fs2ms_{tag}_inf_mel") and gs.err(out[1][0], g, f"fs2ms_{tag}_inf_mel") < TOL
        b = gs.fs2_batch(g, f"fs2ms_{tag}_fwd")
        with torch.no_grad():
            fw = ofs.fs2_forward(p, cfg, b["text"], b["text_lengths"], b["speech_lengths"], b["durations"], b["pitch"], b["energy"],
                                 spk_id=torch.from_numpy(g[f"fs2ms_{tag}_fwd_spk"]), tone_id=torch.from_numpy(g[f"fs2ms_{tag}_fwd_tone"]))
        assert gs.err(fw[1], g, f"fs2ms_{tag}_fwd_after") < TOL
        assert gs.err(fw[2], g, f"fs2ms_{tag}_fwd_d") < TOL
