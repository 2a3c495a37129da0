"""CPU: pin the oracle restatement to the reference's own outputs.

tests/golden/*.npz were produced by the UNMODIFIED reference (oracle/gen_golden.py); the oracle must reproduce them.
fp32 oracle vs reference: same ATen kernels -> bit-identical at one thread; a few ulp otherwise (thread-count dependent
reduction order, SURVEY.md Appendix D)."""
import json
import os

import numpy as np
import pytest
import torch

from fastspeech2_b200 import configs, synth
from oracle import fs2_oracle as O
from oracle.gen_golden import golden_sample

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name,ds", [("fs2_lj", "LJSpeech"), ("fs2_libri", "LibriTTS")])
def test_acoustic_oracle_reproduces_reference_outputs(name, ds, scratch):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    pc, mc = configs.make_configs(ds, scratch)
    sd = synth.fastspeech2_state_dict(pc, mc, seed=int(z["seed"]))
    t = lambda k: torch.from_numpy(z[k])
    out = O.fastspeech2_forward(sd, t("speakers"), t("texts"), t("src_lens"), int(z["max_src_len"]),
                                p_control=float(z["p_control"]), e_control=float(z["e_control"]), d_control=float(z["d_control"]))
    assert torch.equal(out[5], t("d_rounded")) and torch.equal(out[9], t("mel_lens"))
    assert torch.equal(out[6], t("src_masks")) and torch.equal(out[7], t("mel_masks"))
    for i, k in ((0, "mel"), (1, "postnet_mel"), (2, "p_pred"), (3, "e_pred"), (4, "logd")):
        assert (out[i] - t(k)).abs().max() < 5e-6, k
    # fp64 evaluation of the same restatement: bounds the fp32 noise of the reference itself
    out64 = O.fastspeech2_forward(sd, t("speakers"), t("texts"), t("src_lens"), int(z["max_src_len"]), dtype=torch.float64,
                                  p_control=float(z["p_control"]), e_control=float(z["e_control"]), d_control=float(z["d_control"]))
    assert torch.equal(out64[9], t("mel_lens"))
    assert (out64[1].float() - t("postnet_mel")).abs().max() < 2e-5


def test_acoustic_oracle_reproduces_reference_outputs_paper_config(scratch):
    """config/LJSpeech_paper: 4-layer decoder, frame-level pitch / energy, log-spaced pitch edges (model/modules.py:48-54,:139-148)."""
    from oracle.gen_golden import paper_state_dict
    z = np.load(os.path.join(GOLD, "fs2_lj_paper.npz"))
    pc, mc = configs.make_configs("LJSpeech_paper", scratch)
    sd = paper_state_dict(pc, mc, int(z["seed"]))
    assert sum(k.endswith("slf_attn.fc.bias") for k in sd if k.startswith("decoder.")) == 4
    edges = sd["variance_adaptor.pitch_bins"]
    assert not torch.allclose(edges[1:] - edges[:-1], (edges[1] - edges[0]).expand(edges.numel() - 1))     # log-spaced
    t = lambda k: torch.from_numpy(z[k])
    out = O.fastspeech2_forward(sd, t("speakers"), t("texts"), t("src_lens"), int(z["max_src_len"]), p_control=float(z["p_control"]),
                                pitch_level="frame_level", energy_level="frame_level")
    assert torch.equal(out[5], t("d_rounded")) and torch.equal(out[9], t("mel_lens")) and torch.equal(out[7], t("mel_masks"))
    assert out[2].shape == t("p_pred").shape == out[0].shape[:2]
    for i, k in ((0, "mel"), (1, "postnet_mel"), (4, "logd")):
        assert (out[i] - t(k)).abs().max() < 5e-6, k
    for i, k in ((2, "p_pred"), (3, "e_pred")):     # raw-valued (hundreds; head weights x100..250 amplify the thread-count noise): relative
        assert ((out[i] - t(k)).abs() / (1 + t(k).abs())).max() < 5e-5, k


@pytest.mark.parametrize("name", ["LJSpeech", "universal"])
def test_vocoder_oracle_reproduces_reference_outputs_real_checkpoint(name):
    """The shipped generator weights (hifigan/generator_*.pth.tar.zip): oracle vs the unmodified reference's committed output."""
    from oracle import real_ckpt
    sd = real_ckpt.load(name)
    if sd is None and os.path.exists(real_ckpt.source_zip(name)):
        sd = real_ckpt.read_reference_checkpoint(name)
    if sd is None:
        pytest.skip("real checkpoint fixture not present (run __graft_entry__.build() where /root/reference exists)")
    z = np.load(os.path.join(GOLD, f"hifigan_real_{name}.npz"))
    wav = O.hifigan_forward(sd, torch.from_numpy(z["mel"]))
    assert (wav - torch.from_numpy(z["wav"])).abs().max() < 2e-6


def test_vocoder_oracle_reproduces_reference_outputs():
    z = np.load(os.path.join(GOLD, "hifigan.npz"))
    sd = synth.hifigan_state_dict(configs.HIFIGAN_CONFIG, seed=int(z["seed"]))
    wav = O.hifigan_forward(sd, torch.from_numpy(z["mel"]))
    assert wav.shape == z["wav"].shape
    assert (wav - torch.from_numpy(z["wav"])).abs().max() < 1e-5


def test_state_dict_key_contract(scratch):
    """Our modules expose exactly the reference's state_dict keys and shapes (checkpoints must load unchanged)."""
    from fastspeech2_b200.hifigan import AttrDict, Generator
    from fastspeech2_b200.model import FastSpeech2
    want = json.load(open(os.path.join(GOLD, "state_dict_keys.json")))
    for ds in ("LJSpeech", "LibriTTS", "LJSpeech_paper"):
        pc, mc = configs.make_configs(ds, scratch)
        got = {k: list(v.shape) for k, v in FastSpeech2(pc, mc).state_dict().items()}
        assert got == want[ds]
    gen = Generator(AttrDict(configs.HIFIGAN_CONFIG))
    assert {k: list(v.shape) for k, v in gen.state_dict().items()} == want["hifigan_weight_norm"]
    gen.eval()
    gen.remove_weight_norm()
    assert {k: list(v.shape) for k, v in gen.state_dict().items()} == want["hifigan_folded"]


def test_remove_weight_norm_matches_oracle_fold():
    from fastspeech2_b200.hifigan import AttrDict, Generator
    sd = synth.hifigan_state_dict(configs.HIFIGAN_CONFIG, seed=5)
    gen = Generator(AttrDict(configs.HIFIGAN_CONFIG))
    gen.load_state_dict(sd)
    gen.eval()
    gen.remove_weight_norm()
    folded = O.fold_weight_norm(sd)
    for k, v in gen.state_dict().items():
        assert torch.allclose(v, folded[k], rtol=1e-6, atol=1e-8), k


def _assert_pinned(z, prefix, out, tol=5e-6):
    for i in range(5):
        assert tuple(out[i].shape) == tuple(z[f"{prefix}{i}_shape"]), (prefix, i)
        assert np.abs(golden_sample(out[i].numpy()) - z[f"{prefix}{i}"]).max() < tol, (prefix, i)


def test_oracle_vs_live_reference(scratch):
    """LibriTTS with pitch / duration control, the teacher-forced path on the reference's own predictions, and a second
    random-weight Generator: oracle vs the outputs the unmodified reference recorded (oracle/gen_golden.py gen_pins)."""
    z = np.load(os.path.join(GOLD, "oracle_pins_libri.npz"))
    pc, mc = configs.make_configs("LibriTTS", scratch)
    sd = synth.fastspeech2_state_dict(pc, mc, seed=int(z["seed"]))
    t = lambda k: torch.from_numpy(z[k])
    spk, texts, lens, L = t("speakers"), t("texts"), t("src_lens"), int(z["max_src_len"])
    got = O.fastspeech2_forward(sd, spk, texts, lens, L, p_control=0.9, d_control=1.2)
    assert torch.equal(got[9], t("mel_lens")) and torch.equal(got[5], t("d_rounded"))
    _assert_pinned(z, "out", got)
    # teacher-forced path
    ml = t("mel_lens")
    got2 = O.fastspeech2_forward(sd, spk, texts, lens, L, None, ml, int(ml.max()), t("p_pred"), t("e_pred"), t("d_rounded").long())
    _assert_pinned(z, "teacher", got2)
    hsd = synth.hifigan_state_dict(configs.HIFIGAN_CONFIG, seed=int(z["hifigan_seed"]))
    wav = O.hifigan_forward(hsd, t("hifigan_mel"))
    assert tuple(wav.shape) == tuple(z["wav_shape"])
    assert np.abs(golden_sample(wav.numpy()) - z["wav"]).max() < 1e-5


def test_oracle_frame_level_vs_live_reference(scratch):
    """frame_level pitch / energy (config/LJSpeech_paper, model/modules.py:139-148): oracle vs the outputs the unmodified reference
    recorded (oracle/gen_golden.py gen_pins)."""
    import copy
    z = np.load(os.path.join(GOLD, "oracle_pins_frame_level.npz"))
    pc, mc = configs.make_configs("LJSpeech", scratch)
    pc = copy.deepcopy(pc)
    pc["preprocessing"]["pitch"]["feature"] = "frame_level"
    pc["preprocessing"]["energy"]["feature"] = "frame_level"
    sd = synth.fastspeech2_state_dict(pc, mc, seed=int(z["seed"]))
    t = lambda k: torch.from_numpy(z[k])
    got = O.fastspeech2_forward(sd, t("speakers"), t("texts"), t("src_lens"), int(z["max_src_len"]), p_control=float(z["p_control"]),
                                pitch_level="frame_level", energy_level="frame_level")
    assert torch.equal(got[9], t("mel_lens")) and torch.equal(got[5], t("d_rounded")) and got[2].shape == got[0].shape[:2]
    _assert_pinned(z, "out", got)
