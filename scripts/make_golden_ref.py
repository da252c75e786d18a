"""Golden vectors produced by EXECUTING THE REFERENCE'S OWN PYTHON for the hot path.

PaddlePaddle cannot be installed in the build container, so the reference cannot run as is.  Its model code is plain Python
that calls ~60 Paddle primitives; `scripts/refexec/paddle_standin.py` maps those primitives onto torch (same mathematical
definitions; the few Paddle-specific semantics are the ones oracle/README.md lists), `scripts/refexec/loader.py` imports the
reference's files from a checkout of it without running `parakeet/__init__.py`.  Under that stand-in this script builds the
reference's own FastSpeech2 / PWGGenerator / ConditionalWaveFlow classes, loads the oracle's seeded Paddle-layout state dicts
into them (which also checks every state-dict key and shape against the reference's class tree) and records what the
REFERENCE code computes.  tests/test_oracle_cpu.py then holds the oracle to these vectors.  Large arrays are stored as
samples (tests/golden_sample.py) to keep the vectors small.

    python scripts/make_golden_ref.py REFERENCE_DIR    # a PaddlePaddle/Parakeet checkout; writes tests/golden/ref_executed*.npz
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from golden_sample import compact  # noqa: E402
from refexec import loader, paddle_standin  # noqa: E402

REF = None            # <REFERENCE_DIR>/parakeet, set by main()
GOLD = os.path.join(ROOT, "tests", "golden")
T = paddle_standin.T


def load_by_path(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def small_pieces(out):
    # numpy-only collate padding (parakeet/data/batch.py:170-189)
    batch = load_by_path(os.path.join(REF, "data", "batch.py"), "ref_batch")
    rng = np.random.RandomState(20260923)
    lengths = [5, 11, 3, 8]
    seqs = {"text": [rng.randint(1, 70, size=n).astype(np.int64) for n in lengths],
            "speech": [rng.randn(3 * n, 7).astype(np.float32) for n in lengths],
            "pitch": [rng.randn(n, 1).astype(np.float32) for n in lengths]}
    for name, ss in seqs.items():
        for i, s in enumerate(ss):
            out[f"{name}_in{i}"] = s
        out[f"{name}_out"] = batch.batch_sequences(ss)
    out["n"] = np.asarray(len(lengths))
    # padding masks (modules/nets_utils.py:54-125) and the length regulator (fastspeech2_predictor/length_regulator.py:46-89)
    from parakeet.modules import nets_utils as nets
    from parakeet.modules.fastspeech2_predictor.length_regulator import LengthRegulator
    for i, lens in enumerate(([5, 3, 2], [1], [7, 7, 4, 9])):
        out[f"mask_len{i}"] = np.asarray(lens, dtype=np.int64)
        out[f"mask_pad{i}"] = nets.make_pad_mask(T(torch.tensor(lens))).numpy()
        out[f"mask_nonpad{i}"] = nets.make_non_pad_mask(lens).numpy()
    lr = LengthRegulator()
    rng = np.random.RandomState(7)
    cases = {"a": ([[1, 2, 2, 1], [3, 1, 4, 0]], 3),                                  # tests/unit/test_expansion.py:20-24
             "b": (rng.randint(0, 6, size=(3, 17)).tolist(), 8), "c": ([[0, 0, 5], [2, 0, 0]], 4)}
    for name, (ds, c) in cases.items():
        d = np.asarray(ds, dtype=np.int64)
        x = rng.randn(d.shape[0], d.shape[1], c).astype(np.float32)
        y = lr(T(torch.from_numpy(x)), T(torch.from_numpy(d)))
        out[f"lr_{name}_x"], out[f"lr_{name}_d"], out[f"lr_{name}_y"] = x, d, y.numpy()


def check_keys(ref, params, what):
    own = dict(ref.named_parameters())
    own.update(dict(ref.named_buffers()))
    own = {k: v for k, v in own.items() if "generated_tensor_" not in k}
    missing, extra = [k for k in own if k not in params], [k for k in params if k not in own]
    bad = [k for k in own if k in params and tuple(own[k].shape) != tuple(params[k].shape)]
    assert not missing and not extra and not bad, (what, missing[:5], extra[:5], bad[:5])
    return sorted(own)


def fastspeech2(out):
    from oracle import fastspeech2 as ofs
    from parakeet.models.fastspeech2.fastspeech2 import FastSpeech2, FastSpeech2Loss
    cfg = dict(ofs.LJSPEECH_MODEL_CFG)
    ref = FastSpeech2(idim=80, odim=80, **cfg)
    ref.eval()
    params = ofs.synth_params(1)
    out["fs2_keys"] = np.asarray(check_keys(ref, params, "FastSpeech2"))
    ref.set_state_dict(params)
    with torch.no_grad():
        xs, _ = ofs.synth_text(1, [100])                                               # cfg1
        out["fs2_inf_text"] = xs[0].numpy()
        out["fs2_inf_mel"] = ref.inference(T(xs[0])).numpy()
        out["fs2_inf_mel_alpha"] = ref.inference(T(xs[0]), alpha=1.3).numpy()        # uses the stand-in's round (restated)
        b = ofs.synth_train_batch(5, [23, 31, 17])
        out["fs2_fwd_seed"] = np.asarray(5)
        for k, v in b.items():
            out[f"fs2_fwd_{k}"] = v.numpy()
        before, after, d_outs, p_outs, e_outs, ys, olens = ref(T(b["text"]), T(b["text_lengths"]), T(b["speech"]), T(b["speech_lengths"]),
                                                               T(b["durations"]), T(b["pitch"]), T(b["energy"]))
        for k, v in (("before", before), ("after", after), ("d_outs", d_outs), ("p_outs", p_outs), ("e_outs", e_outs)):
            out[f"fs2_fwd_out_{k}"] = v.numpy()
        crit = FastSpeech2Loss(use_masking=True, use_weighted_masking=False)
        l1, dur, pitch, energy = crit(after_outs=after, before_outs=before, d_outs=d_outs, p_outs=p_outs, e_outs=e_outs, ys=ys,
                                      ds=T(b["durations"]), ps=T(b["pitch"]), es=T(b["energy"]), ilens=T(b["text_lengths"]), olens=olens)
        out["fs2_loss"] = np.asarray([float(l1), float(dur), float(pitch), float(energy)], dtype=np.float64)


def fastspeech2_multispeaker(out):
    """The aishell3 / vctk shape of the model (conf/default.yaml:76-77: spk_embed_dim 256, concat) plus tone embeddings ("add"):
    the reference's own inference(spk_id, tone_id) and batched forward(..., spk_id, tone_id) - including its F.normalize(axis=1)
    over TIME for the batched (B, T, D) tone embeddings."""
    from oracle import fastspeech2 as ofs
    from parakeet.models.fastspeech2.fastspeech2 import FastSpeech2
    for tag, (st, tt) in (("a", ("concat", "add")), ("b", ("add", "concat"))):
        cfg = dict(ofs.LJSPEECH_MODEL_CFG, num_speakers=6, spk_embed_dim=256, spk_embed_integration_type=st, num_tones=7, tone_embed_dim=32,
                   tone_embed_integration_type=tt)
        ref = FastSpeech2(idim=80, odim=80, **cfg)
        ref.eval()
        params = ofs.add_speaker_tone_params(ofs.synth_params(1), 1, spk_type=st, tone_type=tt)
        out[f"fs2ms_{tag}_keys"] = np.asarray(check_keys(ref, params, "FastSpeech2(multi-speaker)"))
        ref.set_state_dict(params)
        g = torch.Generator().manual_seed(77)
        with torch.no_grad():
            xs, _ = ofs.synth_text(21, [37])
            tone = torch.randint(0, 7, (37,), generator=g)
            spk = torch.tensor([4])
            out[f"fs2ms_{tag}_inf_text"], out[f"fs2ms_{tag}_inf_tone"] = xs[0].numpy(), tone.numpy()
            # tone "concat" cannot run through the reference's inference(): it expands the (T, D) embeddings with
            # shape=[-1, T, -1], a -1 in a dimension that does not exist (fastspeech2.py:611-612) - speaker only there
            out[f"fs2ms_{tag}_inf_mel"] = ref.inference(T(xs[0]), spk_id=T(spk), tone_id=T(tone) if tt == "add" else None).numpy()
            b = ofs.synth_train_batch(22, [14, 19])
            out[f"fs2ms_{tag}_fwd_seed"] = np.asarray(22)
            tone_b = torch.randint(0, 7, tuple(b["text"].shape), generator=g)
            spk_b = torch.tensor([1, 5])
            for k, v in b.items():
                out[f"fs2ms_{tag}_fwd_{k}"] = v.numpy()
            out[f"fs2ms_{tag}_fwd_tone"], out[f"fs2ms_{tag}_fwd_spk"] = tone_b.numpy(), spk_b.numpy()
            res = ref(T(b["text"]), T(b["text_lengths"]), T(b["speech"]), T(b["speech_lengths"]), T(b["durations"]), T(b["pitch"]),
                      T(b["energy"]), tone_id=T(tone_b), spk_id=T(spk_b))
            out[f"fs2ms_{tag}_fwd_after"], out[f"fs2ms_{tag}_fwd_d"] = res[1].numpy(), res[2].numpy()


def fastspeech2_training(out):
    """The reference model in TRAIN mode (dropout rates set to 0, BatchNorm on batch statistics), its own FastSpeech2Loss, the
    sum of the four losses as in fastspeech2_updater.py:83, torch autograd through the reference's code: the gradients the
    CUDA training step is checked against (via the oracle), now produced by the reference's wiring."""
    from oracle import fastspeech2 as ofs
    from parakeet.models.fastspeech2.fastspeech2 import FastSpeech2, FastSpeech2Loss
    zero = dict(transformer_enc_dropout_rate=0.0, transformer_enc_positional_dropout_rate=0.0, transformer_enc_attn_dropout_rate=0.0,
                transformer_dec_dropout_rate=0.0, transformer_dec_positional_dropout_rate=0.0, transformer_dec_attn_dropout_rate=0.0,
                duration_predictor_dropout_rate=0.0, postnet_dropout_rate=0.0, pitch_predictor_dropout=0.0, pitch_embed_dropout=0.0,
                energy_predictor_dropout=0.0, energy_embed_dropout=0.0, stop_gradient_from_pitch_predictor=True,
                stop_gradient_from_energy_predictor=False)
    ref = FastSpeech2(idim=80, odim=80, **ofs.LJSPEECH_MODEL_CFG, **zero)
    ref.train()
    params = ofs.synth_params(1)
    ref.set_state_dict(params)
    b = ofs.synth_train_batch(9, [19, 27, 22])
    out["fs2_train_seed"] = np.asarray(9)
    for k, v in b.items():
        out[f"fs2_train_{k}"] = v.numpy()
    before, after, d_outs, p_outs, e_outs, ys, olens = ref(T(b["text"]), T(b["text_lengths"]), T(b["speech"]), T(b["speech_lengths"]),
                                                           T(b["durations"]), T(b["pitch"]), T(b["energy"]))
    l1, dur, pitch, energy = FastSpeech2Loss()(after_outs=after, before_outs=before, d_outs=d_outs, p_outs=p_outs, e_outs=e_outs, ys=ys,
                                               ds=T(b["durations"]), ps=T(b["pitch"]), es=T(b["energy"]), ilens=T(b["text_lengths"]),
                                               olens=olens)
    (l1 + dur + pitch + energy).backward()
    out["fs2_train_loss"] = np.asarray([float(l1), float(dur), float(pitch), float(energy)], dtype=np.float64)
    # a representative subset of gradients (all 198 would be 150 MB): every kind of tensor on the path, + the L2 norm of each
    keep = ["encoder.embed.0.weight", "encoder.embed.1.alpha", "encoder.encoders.0.self_attn.linear_q.weight",
            "encoder.encoders.3.feed_forward.w_1.weight", "encoder.encoders.2.norm1.bias", "encoder.after_norm.weight",
            "duration_predictor.conv.0.0.weight", "duration_predictor.linear.bias", "pitch_predictor.conv.4.0.bias",
            "pitch_embed.0.weight", "energy_embed.0.bias", "decoder.embed.0.alpha", "decoder.encoders.1.self_attn.linear_out.weight",
            "decoder.encoders.3.feed_forward.w_2.bias", "feat_out.weight", "postnet.postnet.0.0.weight", "postnet.postnet.2.1.weight",
            "postnet.postnet.4.1.bias"]
    named = dict(ref.named_parameters())
    for k in keep:
        gk = named[k].grad
        gk = (gk if gk is not None else torch.zeros_like(named[k])).detach()
        out["fs2_train_grad/" + k] = gk.numpy()
        out["fs2_train_gradnorm/" + k] = np.asarray(float(gk.double().norm()))
    bufs = dict(ref.named_buffers())
    for k in ("postnet.postnet.0.1._mean", "postnet.postnet.0.1._variance", "postnet.postnet.4.1._variance"):
        out["fs2_train_stat/" + k] = bufs[k].detach().numpy()


def parallel_wavegan(out):
    from oracle import pwg as opwg
    from parakeet.models.parallel_wavegan.parallel_wavegan import PWGGenerator
    cfg = dict(opwg.DEFAULT_GENERATOR_PARAMS)
    cfg["use_weight_norm"] = False                                                    # the folded weights are loaded
    ref = PWGGenerator(**cfg)
    ref.eval()
    folded = opwg.fold_weight_norm(opwg.synth_params(2, weight_norm=True))
    out["pwg_keys"] = np.asarray(check_keys(ref, folded, "PWGGenerator"))
    ref.set_state_dict(folded)
    x, c = opwg.synth_inputs(2, batch=2, mel_frames=10)
    with torch.no_grad():
        out["pwg_x"], out["pwg_c"] = x.numpy(), c.numpy()
        out["pwg_y"] = ref(T(x), T(c)).numpy()
    # with weight norm applied by the reference's own apply_weight_norm: the g / v parametrisation and its 1-D weight_g
    cfg["use_weight_norm"] = True
    ref2 = PWGGenerator(**cfg)
    ref2.eval()
    wn = opwg.synth_params(2, weight_norm=True)
    out["pwg_wn_keys"] = np.asarray(check_keys(ref2, wn, "PWGGenerator(weight_norm)"))
    ref2.set_state_dict(wn)
    with torch.no_grad():
        out["pwg_y_weight_norm"] = ref2(T(x), T(c)).numpy()


def pwg_discriminator(out):
    from oracle import pwg as opwg
    from parakeet.models.parallel_wavegan.parallel_wavegan import PWGDiscriminator
    cfg = dict(opwg.DEFAULT_DISCRIMINATOR_PARAMS)
    cfg["use_weight_norm"] = False
    ref = PWGDiscriminator(**cfg)
    ref.eval()
    dp = opwg.synth_discriminator_params(12)
    out["pwgd_keys"] = np.asarray(check_keys(ref, dp, "PWGDiscriminator"))
    ref.set_state_dict(dp)
    x = torch.randn(2, 1, 900, generator=torch.Generator().manual_seed(21))
    with torch.no_grad():
        out["pwgd_x"], out["pwgd_y"] = x.numpy(), ref(T(x)).numpy()


def waveflow(out):
    from oracle import waveflow as owf
    from parakeet.models.waveflow import ConditionalWaveFlow
    ref = ConditionalWaveFlow(upsample_factors=[16, 16], n_flows=8, n_layers=8, n_group=16, channels=64, n_mels=80, kernel_size=[3, 3])
    ref.eval()
    params = owf.synth_params(4)
    out["wf_keys"] = np.asarray(check_keys(ref, params, "ConditionalWaveFlow"))
    ref.set_state_dict(params)
    g = torch.Generator().manual_seed(4)
    mel = torch.randn(2, 80, 9, generator=g) * 0.5 - 3
    with torch.no_grad():
        cond = ref.encoder(T(mel), trim_conv_artifact=True)
        z = torch.randn(2, cond.shape[-1], generator=g)
        out["wf_mel"], out["wf_z"] = mel.numpy(), z.numpy()
        out["wf_cond"] = cond.numpy()
        out["wf_x"] = ref.decoder.inverse(T(z), cond).numpy()
        # second vector: 22 mel frames -> W = 335 columns > 2 x 128, so the +-128 width taps of layer 7 land on live data
        # (the 9-frame vector above has W = 127: its widest taps only ever see zero padding)
        mel2 = torch.randn(1, 80, 22, generator=g) * 0.5 - 3
        cond2 = ref.encoder(T(mel2), trim_conv_artifact=True)
        z2 = torch.randn(1, cond2.shape[-1], generator=g)
        out["wf2_mel"], out["wf2_z"] = mel2.numpy(), z2.numpy()
        out["wf2_x"] = ref.decoder.inverse(T(z2), cond2).numpy()
    # third vector: the SHIPPED config (examples/waveflow/config.py: 128 residual channels), W = 335 columns
    ref128 = ConditionalWaveFlow(upsample_factors=[16, 16], n_flows=8, n_layers=8, n_group=16, channels=128, n_mels=80, kernel_size=[3, 3])
    ref128.eval()
    params128 = owf.synth_params(5, channels=128)
    check_keys(ref128, params128, "ConditionalWaveFlow(128)")
    ref128.set_state_dict(params128)
    g = torch.Generator().manual_seed(45)
    with torch.no_grad():
        mel3 = torch.randn(1, 80, 22, generator=g) * 0.5 - 3
        cond3 = ref128.encoder(T(mel3), trim_conv_artifact=True)
        z3 = torch.randn(1, cond3.shape[-1], generator=g)
        out["wf128_mel"], out["wf128_z"] = mel3.numpy(), z3.numpy()
        out["wf128_x"] = ref128.decoder.inverse(T(z3), cond3).numpy()


def wrappers_and_stft(out):
    """FastSpeech2Inference / PWGInference (normaliser wrappers, PWG's replicate padding and transposes) and modules/audio.STFT."""
    import paddle
    from oracle import fastspeech2 as ofs
    from oracle import pwg as opwg
    from parakeet.models.fastspeech2.fastspeech2 import FastSpeech2, FastSpeech2Inference
    from parakeet.models.parallel_wavegan.parallel_wavegan import PWGGenerator, PWGInference
    from parakeet.modules.audio import STFT
    from parakeet.modules.normalizer import ZScore
    g = torch.Generator().manual_seed(11)
    mu, sigma = torch.randn(80, generator=g), torch.rand(80, generator=g) + 0.5
    out["wr_mu"], out["wr_sigma"] = mu.numpy(), sigma.numpy()
    fs = FastSpeech2(idim=80, odim=80, **ofs.LJSPEECH_MODEL_CFG)
    fs.eval()
    fs.set_state_dict(ofs.synth_params(1))
    text = torch.randint(1, 79, (20,), generator=g)
    with torch.no_grad():
        logmel = FastSpeech2Inference(ZScore(T(mu), T(sigma)), fs)(T(text))
    out["wr_text"], out["wr_logmel"] = text.numpy(), logmel.numpy()
    cfg = dict(opwg.DEFAULT_GENERATOR_PARAMS)
    cfg["use_weight_norm"] = False
    gen = PWGGenerator(**cfg)
    gen.eval()
    gen.set_state_dict(opwg.fold_weight_norm(opwg.synth_params(2, weight_norm=True)))
    mel = torch.randn(6, 80, generator=g)
    noise = torch.randn(1, 1, 6 * 300, generator=g)
    real_randn = paddle.randn
    paddle.randn = lambda shape, dtype=None: T(noise)                 # inference() draws its own noise: supply ours
    try:
        with torch.no_grad():
            wav = PWGInference(ZScore(T(mu), T(sigma)), gen)(T(mel))
    finally:
        paddle.randn = real_randn
    out["wr_pwg_logmel"], out["wr_pwg_noise"], out["wr_pwg_wav"] = mel.numpy(), noise.numpy(), wav.numpy()
    wavs = torch.randn(2, 3000, generator=g)
    out["stft_x"] = wavs.numpy()
    for tag, (n_fft, hop, win) in (("a", (512, 128, 512)), ("b", (1024, 120, 600))):
        st = STFT(n_fft, hop, win, window="hann")
        with torch.no_grad():
            re, im = st(T(wavs))
            mag = st.magnitude(T(wavs))
        out[f"stft_{tag}_re"], out[f"stft_{tag}_im"], out[f"stft_{tag}_mag"] = re.numpy(), im.numpy(), mag.numpy()
    # MultiResolutionSTFTLoss (modules/stft_loss.py:163-219): paddle.signal.stft mapped to torch.stft; the clipping, the
    # transposes, the Frobenius ratio, the log-magnitude L1 and the mean over resolutions are the reference's code
    from parakeet.modules.stft_loss import MultiResolutionSTFTLoss
    other = torch.randn(2, 3000, generator=g) * 0.3
    out["mrstft_y"] = other.numpy()
    with torch.no_grad():
        sc, mag = MultiResolutionSTFTLoss()(T(wavs), T(other))
    out["mrstft_loss"] = np.asarray([float(sc), float(mag)], dtype=np.float64)


def main():
    global REF
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    REF = os.path.join(os.path.abspath(sys.argv[1]), "parakeet")
    uninstall = loader.install(paddle_standin.build(), os.path.dirname(REF))
    try:
        small, models = {}, {}
        small_pieces(small)
        fastspeech2(models)
        fastspeech2_multispeaker(models)
        fastspeech2_training(models)
        parallel_wavegan(models)
        pwg_discriminator(models)
        waveflow(models)
        wrappers_and_stft(models)
    finally:
        uninstall()
    models = compact(models, keep_full=("pwg_x", "stft_x", "mrstft_y", "wf2_z", "wf128_z"))   # inputs the tests read back
    np.savez(os.path.join(GOLD, "ref_executed.npz"), **small)
    np.savez_compressed(os.path.join(GOLD, "ref_executed_models.npz"), **models)
    for name, d in (("ref_executed.npz", small), ("ref_executed_models.npz", models)):
        print(name, os.path.getsize(os.path.join(GOLD, name)) // 1024, "KB", len(d), "arrays")


if __name__ == "__main__":
    main()
