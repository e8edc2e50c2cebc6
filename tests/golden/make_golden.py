# coding: utf-8
"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

Needs a checkout of the original r9y9/wavenet_vocoder project:

    python tests/golden/make_golden.py <path of the wavenet_vocoder checkout>

For each small case it builds the reference ``WaveNet`` with seeded random weights, runs
  (1) teacher-forced ``incremental_forward`` while spying on the sampler input (the per-step head
      output the public API never returns for scalar-input models, SURVEY.md 8(c) recipe 1),
  (2) the batch ``forward()`` for the reference's own online==offline check
      (tests/test_model.py:330-366),
  (3) free-running seeded ``incremental_forward``, and
  (4) the same over at most 48 steps with another torch seed,
then runs oracle/wavenet_oracle.py on the same weights/inputs/seed, asserts BIT equality with the
reference for (1), (3) and (4), and writes (1)-(3) to ``<case>.npz`` and (4) of every case to
``reference_arm.npz``.  The committed vectors let the oracle and the CUDA path be checked without
the original project.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if len(sys.argv) != 2:
    sys.exit("usage: python tests/golden/make_golden.py <path of the wavenet_vocoder checkout>")
sys.path.insert(0, os.path.abspath(sys.argv[1]))
warnings.filterwarnings("ignore")

import wavenet_vocoder as ref_pkg                      # noqa: E402  (the reference)
from wavenet_vocoder import wavenet as ref_wavenet     # noqa: E402
from oracle import wavenet_oracle as orc               # noqa: E402

CASES = {
    # name: (ctor kwargs, B, T, extras)
    "mulaw_softmax": dict(
        kw=dict(out_channels=256, layers=4, stacks=2, residual_channels=16, gate_channels=32,
                skip_out_channels=16, cin_channels=-1, gin_channels=-1, scalar_input=False,
                dropout=0.0),
        B=2, T=48),
    "mol_cond": dict(
        kw=dict(out_channels=30, layers=6, stacks=2, residual_channels=32, gate_channels=64,
                skip_out_channels=32, cin_channels=8, gin_channels=-1, scalar_input=True,
                output_distribution="Logistic", dropout=0.0),
        B=2, T=80),
    "mol_upsample": dict(
        kw=dict(out_channels=30, layers=6, stacks=3, residual_channels=24, gate_channels=48,
                skip_out_channels=40, cin_channels=8, cin_pad=1, gin_channels=-1, scalar_input=True,
                output_distribution="Logistic", dropout=0.0, upsample_conditional_features=True,
                upsample_params={"upsample_scales": [2, 4], "cin_channels": 8, "cin_pad": 1}),
        B=2, T=64, frames=8 + 2),
    "gauss_speaker": dict(
        kw=dict(out_channels=2, layers=4, stacks=2, residual_channels=16, gate_channels=32,
                skip_out_channels=24, cin_channels=8, gin_channels=4, n_speakers=3,
                use_speaker_embedding=True, scalar_input=True, output_distribution="Normal",
                dropout=0.0),
        B=1, T=64),
    "mixgauss": dict(
        kw=dict(out_channels=6, layers=4, stacks=1, residual_channels=16, gate_channels=32,
                skip_out_channels=16, cin_channels=-1, gin_channels=-1, scalar_input=True,
                output_distribution="Normal", dropout=0.0),
        B=2, T=48),
}
SHORT_SEED = 11


def path_config(kw):
    return orc.PathConfig(
        out_channels=kw["out_channels"], layers=kw["layers"], stacks=kw["stacks"],
        residual_channels=kw["residual_channels"], gate_channels=kw["gate_channels"],
        skip_out_channels=kw["skip_out_channels"], kernel_size=kw.get("kernel_size", 3),
        cin_channels=kw.get("cin_channels", -1), gin_channels=kw.get("gin_channels", -1),
        scalar_input=kw.get("scalar_input", False),
        output_distribution=kw.get("output_distribution", "Logistic"))


class Spy:
    """Record the tensor handed to the sampler each step (wavenet.py:322-335)."""

    def __init__(self):
        self.rec = []
        self._saved = {}

    def __enter__(self):
        for name in ("sample_from_discretized_mix_logistic", "sample_from_mix_gaussian"):
            fn = getattr(ref_wavenet, name)
            self._saved[name] = fn

            def wrapped(y, _fn=fn, **kw):
                self.rec.append(y.detach().clone().view(y.size(0), -1))
                return _fn(y, **kw)
            setattr(ref_wavenet, name, wrapped)
        return self

    def __exit__(self, *a):
        for k, v in self._saved.items():
            setattr(ref_wavenet, k, v)


def make_case(name, spec):
    kw, B, T = spec["kw"], spec["B"], spec["T"]
    cfg = path_config(kw)
    torch.manual_seed(1234)
    model = ref_pkg.WaveNet(**kw).eval()
    # random-init heads give log-scale ~0 (samples saturate at +-1): bias the log-scale rows so
    # the free-running waveform is non-degenerate (SURVEY.md 8(d)); also randomise biases, which
    # the reference initialises to zero, so bias handling is actually exercised.
    with torch.no_grad():
        for n_, p in model.named_parameters():
            if n_.endswith(".bias"):
                p.normal_(0, 0.05)
        if cfg.scalar_input:
            O = cfg.out_channels
            b = model.last_conv_layers[3].bias
            if O == 2:
                b[1] -= 3.0
            else:
                b[2 * (O // 3):] -= 3.0
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    w = orc.weights_from_state_dict(cfg, sd)

    g_ids = g_vec = c_raw = c_up = None
    gen = torch.Generator().manual_seed(99)
    if cfg.cin_channels > 0:
        if kw.get("upsample_conditional_features"):
            c_raw = torch.randn(B, cfg.cin_channels, spec["frames"], generator=gen)
            with torch.no_grad():
                c_up = model.upsample_net(c_raw)
            assert c_up.size(-1) == T, c_up.shape
        else:
            c_up = torch.randn(B, cfg.cin_channels, T, generator=gen)
            c_raw = c_up
    if cfg.gin_channels > 0:
        g_ids = torch.randint(0, kw["n_speakers"], (B, 1), generator=gen)
        g_vec = orc.embed_speaker(w, g_ids)

    # teacher-forcing input
    if cfg.scalar_input:
        x_tf = (torch.rand(B, 1, T, generator=gen) * 2 - 1) * 0.8
    else:
        idx = torch.randint(0, cfg.out_channels, (B, T), generator=gen)
        x_tf = torch.zeros(B, cfg.out_channels, T).scatter_(1, idx.unsqueeze(1), 1.0)

    out = dict(B=B, T=T)
    with torch.no_grad():
        # (1) teacher forced, reference
        torch.manual_seed(7)
        if cfg.scalar_input:
            with Spy() as spy:
                y_tf_ref = model.incremental_forward(test_inputs=x_tf, c=c_raw, g=g_ids, T=T)
            params_ref = torch.stack(spy.rec, dim=-1)                       # (B,O,T)
        else:
            # softmax=False, quantize=False returns the raw head output itself
            params_ref = model.incremental_forward(test_inputs=x_tf, c=c_raw, g=g_ids, T=T,
                                                   softmax=False, quantize=False)
            torch.manual_seed(7)
            y_tf_ref = model.incremental_forward(test_inputs=x_tf, c=c_raw, g=g_ids, T=T)
        # (2) batch forward (online == offline, tests/test_model.py:355-366)
        y_batch = model(x_tf, c=c_raw, g=g_ids, softmax=False)
        diff = (y_batch - params_ref).abs().max().item()
        assert diff < 1e-4, diff
        # (1') teacher forced, oracle
        torch.manual_seed(7)
        rec = []
        y_tf_orc = orc.incremental_forward(cfg, w, test_inputs=x_tf, c=c_up, g=g_vec, T=T,
                                           params_out=rec)
        params_orc = torch.stack(rec, dim=-1)
        assert torch.equal(params_orc, params_ref), (name, (params_orc - params_ref).abs().max())
        assert torch.equal(y_tf_orc, y_tf_ref), name
        noise_tf = orc.predraw_noise(cfg, B, T, 7)
        y_tf_rep = orc.incremental_forward(cfg, w, test_inputs=x_tf, c=c_up, g=g_vec, T=T,
                                           noise=orc.replay_from_predrawn(cfg, noise_tf))
        assert torch.equal(y_tf_rep, y_tf_ref), name
        # (3) free running, seeded
        seed = 2024
        torch.manual_seed(seed)
        y_free_ref = model.incremental_forward(c=c_raw, g=g_ids, T=T)
        torch.manual_seed(seed)
        y_free_orc = orc.incremental_forward(cfg, w, c=c_up, g=g_vec, T=T)
        assert torch.equal(y_free_ref, y_free_orc), name
        # (3') replayed noise reproduces it too
        B_free = y_free_ref.size(0)      # the reference infers B from c / test_inputs only
        noise = orc.predraw_noise(cfg, B_free, T, seed)
        rec2 = []
        y_free_rep = orc.incremental_forward(cfg, w, c=c_up, g=g_vec, T=T,
                                             noise=orc.replay_from_predrawn(cfg, noise),
                                             params_out=rec2)
        assert torch.equal(y_free_ref, y_free_rep), name
        params_free = torch.stack(rec2, dim=-1)
        # (4) free running over at most 48 steps, another seed (the upsample network fixes the length)
        upsample = kw.get("upsample_conditional_features", False)
        T_short = T if upsample else min(T, 48)
        torch.manual_seed(SHORT_SEED)
        y_short_ref = model.incremental_forward(c=c_raw if c_raw is None or upsample else c_raw[..., :T_short],
                                                g=g_ids, T=T_short)
        torch.manual_seed(SHORT_SEED)
        y_short_orc = orc.incremental_forward(cfg, w, c=None if c_up is None else c_up[..., :T_short], g=g_vec,
                                              T=T_short)
        assert torch.equal(y_short_ref, y_short_orc), name

    out.update({"sd." + k: v.numpy() for k, v in sd.items()})
    out.update({"noise." + k: v.numpy() for k, v in noise.items()})
    out.update({"noise_tf." + k: v.numpy() for k, v in noise_tf.items()})
    out["x_tf"] = x_tf.numpy() if cfg.scalar_input else idx.numpy().astype(np.int32)
    out["params_tf"] = params_ref.numpy()
    out["params_free"] = params_free.numpy()
    out["batch_forward_maxdiff"] = np.float32(diff)
    if cfg.scalar_input:
        out["y_tf"] = y_tf_ref.numpy()
        out["y_free"] = y_free_ref.numpy()
    else:
        out["y_tf"] = y_tf_ref.argmax(1).numpy().astype(np.int32)
        out["y_free"] = y_free_ref.argmax(1).numpy().astype(np.int32)
    if c_up is not None:
        out["c_up"] = c_up.numpy()
        out["c_raw"] = c_raw.numpy()
    if g_ids is not None:
        out["g_ids"] = g_ids.numpy()
        out["g_vec"] = g_vec.numpy()
    out["B_free"] = B_free
    out["seed"] = seed
    out["kw"] = np.array(repr(kw))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("%-14s ok  online/offline maxdiff %.2e  |y_free| mean %.3f" %
          (name, diff, float(np.abs(out["y_free"]).mean())))
    return y_short_ref.numpy()


def main():
    # reference's own known answers for the queue geometry (tests/test_misc.py:9-13)
    assert ref_pkg.receptive_field_size(30, 3, 3) == orc.receptive_field_size(30, 3, 3) == 6139
    assert ref_pkg.receptive_field_size(24, 4, 3) == orc.receptive_field_size(24, 4, 3) == 505
    assert ref_pkg.receptive_field_size(12, 2, 3) == orc.receptive_field_size(12, 2, 3) == 253
    assert ref_pkg.receptive_field_size(30, 1, 3, dilation=lambda x: 1) == \
        orc.receptive_field_size(30, 1, 3, dilation=lambda x: 1) == 61
    short = {name: make_case(name, spec) for name, spec in CASES.items()}
    np.savez_compressed(os.path.join(HERE, "reference_arm.npz"), seed=SHORT_SEED, **short)


if __name__ == "__main__":
    main()
