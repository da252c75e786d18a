"""Reading tests/golden/ref_executed_models.npz, which keeps its large arrays as samples (written by scripts/make_golden_ref.py).

An array of more than SAMPLE elements is stored as its values at SAMPLE fixed positions (sample_index), next to
"shape/<name>" (the full shape) and "absmax/<name>" (the max-abs of the full array), so that the comparisons keep the scale
they have against the full array.  The teacher-forcing speech targets of the FastSpeech2 batches are such samples; the full
batch is rebuilt from the seed stored with it."""
import numpy as np
import torch

from conftest import rel_err

SAMPLE = 4096


def sample_index(n):
    """The SAMPLE positions kept of an array of n elements (numpy's RandomState stream is fixed across numpy versions)."""
    return np.sort(np.random.RandomState(n % 2 ** 32).choice(n, SAMPLE, replace=False))


def compact(arrays, keep_full=()):
    """{name: array} -> the stored form: arrays larger than SAMPLE (other than `keep_full`) as samples + shape + max-abs."""
    out = {}
    for k, a in arrays.items():
        a = np.asarray(a)
        if a.size <= SAMPLE or k in keep_full or a.dtype.kind not in "fiu":
            out[k] = a
        else:
            out[k] = a.reshape(-1)[sample_index(a.size)]
            out["shape/" + k] = np.asarray(a.shape, dtype=np.int64)
            out["absmax/" + k] = np.asarray(np.abs(a).max(), dtype=np.float64)
    return out


def shape(g, name):
    return tuple(int(n) for n in g["shape/" + name]) if "shape/" + name in g else g[name].shape


def err(t, g, name):
    """rel_err(t, the golden array `name`); a sampled one is compared at its sampled positions, relative to its full max-abs."""
    if "shape/" + name not in g:
        return rel_err(t, torch.from_numpy(g[name]))
    assert tuple(t.shape) == shape(g, name), (name, tuple(t.shape), shape(g, name))
    t = t.detach().double().cpu().reshape(-1)[torch.from_numpy(sample_index(t.numel()))]
    return ((t - torch.from_numpy(g[name]).double()).abs().max() / max(float(g["absmax/" + name]), 1e-30)).item()


def fs2_batch(g, prefix):
    """The FastSpeech2 batch `prefix` was computed on: oracle.fastspeech2.synth_train_batch at the stored seed and lengths,
    checked element for element against what is stored of it."""
    from oracle import fastspeech2 as ofs
    b = ofs.synth_train_batch(int(g[prefix + "_seed"]), g[prefix + "_text_lengths"].tolist())
    for k, v in b.items():
        assert err(v, g, f"{prefix}_{k}") == 0, (prefix, k)
    return b
