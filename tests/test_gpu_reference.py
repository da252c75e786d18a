"""The CUDA path against vectors computed by the REFERENCE'S OWN CODE (tests/golden/ref_executed_models.npz, written by
scripts/make_golden_ref.py: the reference's model classes executed on a torch-backed stand-in for the Paddle primitives they
call, with the same seeded state dicts these tests load; large arrays stored as samples, tests/golden_sample.py).  Same
structure as the oracle-golden tests of test_gpu_models.py."""
import os

import numpy as np
import pytest
import torch

import golden_sample as gs
from conftest import rel_err

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-3   # north_star: "within 1e-3 rel fp32" (max-abs error / max-abs reference per tensor)


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLD, "ref_executed_models.npz"))


def test_fastspeech2_cuda_vs_executed_reference(cuda, g):
    from oracle import fastspeech2 as ofs
    from parakeet_b200.models import FastSpeech2, FastSpeech2Loss
    m = FastSpeech2(80, 80, **ofs.LJSPEECH_MODEL_CFG, device=cuda)
    m.set_state_dict(ofs.synth_params(1))
    text = torch.from_numpy(g["fs2_inf_text"]).to(cuda)
    out = m.inference(text)
    assert tuple(out.shape) == gs.shape(g, "fs2_inf_mel")                  # integer durations: same number of frames
    assert gs.err(out, g, "fs2_inf_mel") < TOL
    out13 = m.inference(text, alpha=1.3)
    assert tuple(out13.shape) == gs.shape(g, "fs2_inf_mel_alpha") and gs.err(out13, g, "fs2_inf_mel_alpha") < TOL
    b = {k: v.to(cuda) for k, v in gs.fs2_batch(g, "fs2_fwd").items()}
    before, after, d_outs, p_outs, e_outs, ys, olens = m(b["text"], b["text_lengths"], b["speech"], b["speech_lengths"],
                                                          b["durations"], b["pitch"], b["energy"])
    for name, t in zip(("before", "after", "d_outs", "p_outs", "e_outs"), (before, after, d_outs, p_outs, e_outs)):
        assert gs.err(t, g, f"fs2_fwd_out_{name}") < TOL, name
    losses = FastSpeech2Loss(device=cuda)(after, before, d_outs, p_outs, e_outs, ys, b["durations"], b["pitch"], b["energy"],
                                          b["text_lengths"], olens)
    got = [float(v) for v in losses]
    assert np.allclose(got[:4], g["fs2_loss"], rtol=1e-3), (got, g["fs2_loss"])


def test_pwg_cuda_vs_executed_reference(cuda, g):
    from oracle import pwg as opwg
    from parakeet_b200.models import PWGGenerator
    gen = PWGGenerator(**opwg.DEFAULT_GENERATOR_PARAMS, device=cuda)
    gen.set_state_dict(opwg.synth_params(2, weight_norm=True))
    y = gen(torch.from_numpy(g["pwg_x"]).to(cuda), torch.from_numpy(g["pwg_c"]).to(cuda))
    assert gs.err(y, g, "pwg_y") < TOL
    assert gs.err(y, g, "pwg_y_weight_norm") < TOL                              # the reference's own weight_norm(g, v) path


def test_waveflow_cuda_vs_executed_reference(cuda, g):
    from oracle import waveflow as owf
    from parakeet_b200.models import ConditionalWaveFlow
    wf = ConditionalWaveFlow([16, 16], 8, 8, 16, 64, 80, (3, 3), device=cuda)
    wf.set_state_dict(owf.synth_params(4))
    mel, z = torch.from_numpy(g["wf_mel"]).to(cuda), torch.from_numpy(g["wf_z"]).to(cuda)
    assert gs.err(wf.encode(mel), g, "wf_cond") < 1e-4
    out = wf.infer(mel, z=z)
    assert tuple(out.shape) == gs.shape(g, "wf_x") and gs.err(out, g, "wf_x") < TOL
    # W = 335 columns: the +-128 taps of the widest layer are inside the row (the vector above has W = 127)
    mel2, z2 = torch.from_numpy(g["wf2_mel"]).to(cuda), torch.from_numpy(g["wf2_z"]).to(cuda)
    out2 = wf.infer(mel2, z=z2)
    assert tuple(out2.shape) == gs.shape(g, "wf2_x") and gs.err(out2, g, "wf2_x") < TOL
    # the reference's shipped config (examples/waveflow/config.py: 128 residual channels), W = 335
    wf128 = ConditionalWaveFlow([16, 16], 8, 8, 16, 128, 80, (3, 3), device=cuda)
    wf128.set_state_dict(owf.synth_params(5, channels=128))
    mel3, z3 = torch.from_numpy(g["wf128_mel"]).to(cuda), torch.from_numpy(g["wf128_z"]).to(cuda)
    out3 = wf128.infer(mel3, z=z3)
    assert tuple(out3.shape) == gs.shape(g, "wf128_x") and gs.err(out3, g, "wf128_x") < TOL


def test_fs2_multispeaker_tone_cuda_vs_executed_reference(cuda, g):
    """FastSpeech2 with speaker + tone conditioning (both integration types) on the CUDA path against the vectors the
    reference's own code produced: inference(spk_id, tone_id), batched forward, and batch_inference == per-utterance inference."""
    from oracle import fastspeech2 as ofs
    from parakeet_b200.models import FastSpeech2
    for tag, (st, tt) in (("a", ("concat", "add")), ("b", ("add", "concat"))):
        p = ofs.add_speaker_tone_params(ofs.synth_params(1), 1, spk_type=st, tone_type=tt)
        m = FastSpeech2(80, 80, **ofs.LJSPEECH_MODEL_CFG, num_speakers=6, spk_embed_dim=256, spk_embed_integration_type=st, num_tones=7,
                        tone_embed_dim=32, tone_embed_integration_type=tt, device=cuda)
        assert sorted(m.state_dict()) == list(g[f"fs2ms_{tag}_keys"])
        m.set_state_dict(p)
        text, tone = torch.from_numpy(g[f"fs2ms_{tag}_inf_text"]).to(cuda), torch.from_numpy(g[f"fs2ms_{tag}_inf_tone"]).to(cuda)
        spk = torch.tensor([4], device=cuda)
        mel = m.inference(text, spk_id=spk, tone_id=tone if tt == "add" else None)
        assert tuple(mel.shape) == gs.shape(g, f"fs2ms_{tag}_inf_mel") and gs.err(mel, g, f"fs2ms_{tag}_inf_mel") < TOL
        b = {k: v.to(cuda) for k, v in gs.fs2_batch(g, f"fs2ms_{tag}_fwd").items()}
        o = m(b["text"], b["text_lengths"], b["speech"], b["speech_lengths"], b["durations"], b["pitch"], b["energy"],
              tone_id=torch.from_numpy(g[f"fs2ms_{tag}_fwd_tone"]).to(cuda), spk_id=torch.from_numpy(g[f"fs2ms_{tag}_fwd_spk"]).to(cuda))
        assert gs.err(o[1], g, f"fs2ms_{tag}_fwd_after") < TOL
        assert gs.err(o[2], g, f"fs2ms_{tag}_fwd_d") < TOL
        if tt == "add":      # ragged batch == the utterances one by one (per-utterance tone normalisation)
            lengths = [37, 21]
            ids = torch.zeros(2, 37, dtype=torch.int64, device=cuda)
            tones = torch.zeros(2, 37, dtype=torch.int64, device=cuda)
            ids[0], tones[0] = text, tone
            ids[1, :21], tones[1, :21] = text[5:26], tone[3:24]
            spk2 = torch.tensor([4, 2], device=cuda)
            melb, olens, _ = m.batch_inference(ids, torch.tensor(lengths, device=cuda), spk_id=spk2, tone_id=tones)
            assert gs.err(melb[0, :int(olens[0])], g, f"fs2ms_{tag}_inf_mel") < TOL
            one = m.inference(ids[1, :21], spk_id=spk2[1:], tone_id=tones[1, :21])
            assert one.shape[0] == int(olens[1]) and rel_err(melb[1, :int(olens[1])], one) < 1e-4
