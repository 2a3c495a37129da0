"""Generate tests/golden/* by running the UNMODIFIED reference (imported read-only from $FS2_REFERENCE) on CPU.

Run where the reference tree exists:  python -m oracle.gen_golden [base] [pins] [frontend]   (no argument: all three)
The fixtures hold inputs and the reference's OUTPUTS only; weights are regenerated from the seed by
fastspeech2_b200.synth (a pure function of the spec and seed), loaded into the reference with load_state_dict(strict).
The reference ships no golden vectors of its own (SURVEY.md section 4), so these files are the pin.
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fastspeech2_b200 import configs, synth  # noqa: E402
from oracle import ref_import  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def paper_state_dict(pc, mc, seed):
    """LJSpeech_paper weights: the unnormalised pitch / energy predictors are steered into their (raw-valued) bin ranges so that the
    log-spaced pitch edges and many distinct buckets are exercised."""
    sd = synth.fastspeech2_state_dict(pc, mc, seed=seed)
    sd["variance_adaptor.pitch_predictor.linear_layer.bias"].fill_(220.0)
    sd["variance_adaptor.pitch_predictor.linear_layer.weight"] *= 250
    sd["variance_adaptor.energy_predictor.linear_layer.bias"].fill_(60.0)
    sd["variance_adaptor.energy_predictor.linear_layer.weight"] *= 100
    return sd


def golden_sample(a, k: int = 2048) -> np.ndarray:
    """A fixed subset of a flattened array: every element when it has at most `k`, else `k` evenly spaced ones (the spacing is not a
    whole number, so the sample walks across the channel dimension).  Keeps the pins small; the tests take the same subset."""
    a = np.asarray(a).reshape(-1)
    if a.size <= k:
        return a.copy()
    return a[np.linspace(0, a.size - 1, k).astype(np.int64)]


def _save_outputs(d: dict, prefix: str, out):
    for i in range(5):
        d[f"{prefix}{i}"] = golden_sample(out[i].numpy())
        d[f"{prefix}{i}_shape"] = np.array(out[i].shape)


def gen_pins(FastSpeech2, hifigan, tmp):
    """Oracle pins beyond the base fixtures: LibriTTS with pitch / duration control, the teacher-forced path on the reference's own
    predictions, a second random-weight Generator, and LJSpeech with frame-level pitch / energy."""
    import copy
    pc, mc = configs.make_configs("LibriTTS", tmp)
    sd = synth.fastspeech2_state_dict(pc, mc, seed=31)
    ref = FastSpeech2(pc, mc)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    spk, texts, lens, L = synth.make_batch(3, 36, seed=32, n_speakers=904, min_len=10)
    with torch.no_grad():
        want = ref(spk, texts, lens, L, p_control=0.9, d_control=1.2)
        ml = want[9]
        want2 = ref(spk, texts, lens, L, None, ml, int(ml.max()), want[2], want[3], want[5].long())
    d = dict(seed=31, speakers=spk.numpy(), texts=texts.numpy(), src_lens=lens.numpy(), max_src_len=L,
             p_pred=want[2].numpy(), e_pred=want[3].numpy(), d_rounded=want[5].numpy(), mel_lens=want[9].numpy())
    _save_outputs(d, "out", want)
    _save_outputs(d, "teacher", want2)
    h = hifigan.AttrDict(configs.HIFIGAN_CONFIG)
    gen = hifigan.Generator(h)
    gen.load_state_dict(synth.hifigan_state_dict(h, seed=33), strict=True)
    gen.eval()
    gen.remove_weight_norm()
    mel = synth.make_mel(1, 30, seed=34)
    with torch.no_grad():
        wav = gen(mel)
    d.update(hifigan_seed=33, hifigan_mel=mel.numpy(), wav=golden_sample(wav.numpy()), wav_shape=np.array(wav.shape))
    np.savez_compressed(os.path.join(OUT, "oracle_pins_libri.npz"), **d)
    print("oracle_pins_libri mel", tuple(want[0].shape), "mel_lens", want[9].tolist())

    pc, mc = configs.make_configs("LJSpeech", tmp)
    pc = copy.deepcopy(pc)
    pc["preprocessing"]["pitch"]["feature"] = "frame_level"
    pc["preprocessing"]["energy"]["feature"] = "frame_level"
    sd = synth.fastspeech2_state_dict(pc, mc, seed=41)
    ref = FastSpeech2(pc, mc)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    spk, texts, lens, L = synth.make_batch(2, 22, seed=42, min_len=13)
    with torch.no_grad():
        want = ref(spk, texts, lens, L, p_control=1.2)
    d = dict(seed=41, speakers=spk.numpy(), texts=texts.numpy(), src_lens=lens.numpy(), max_src_len=L, p_control=1.2,
             d_rounded=want[5].numpy(), mel_lens=want[9].numpy())
    _save_outputs(d, "out", want)
    np.savez_compressed(os.path.join(OUT, "oracle_pins_frame_level.npz"), **d)
    print("oracle_pins_frame_level mel", tuple(want[0].shape), "mel_lens", want[9].tolist())


FRONTEND_DATASETS = ("LJSpeech", "LibriTTS", "AISHELL3")


def gen_frontend():
    """Every 8th line of the `preprocessed_data/*/val.txt` files the reference ships (64 utterances, 8 batches each) through the
    reference's TextDataset + DataLoader(batch_size=8): the lines, the speaker ids they use, the cleaners, each utterance's phoneme ids
    and the collated batches."""
    import yaml
    from torch.utils.data import DataLoader
    cwd = os.getcwd()
    os.chdir(ref_import.REFERENCE_ROOT)        # the reference's configs hold paths relative to its tree
    try:
        from dataset import TextDataset
        d = {}
        for ds in FRONTEND_DATASETS:
            pc = yaml.safe_load(open(f"config/{ds}/preprocess.yaml"))
            pre = pc["path"]["preprocessed_path"]
            lines = open(os.path.join(pre, "val.txt"), encoding="utf-8").read().splitlines()[::8]
            src = os.path.join(tempfile.mkdtemp(), "val.txt")
            with open(src, "w", encoding="utf-8") as f:
                f.write("\n".join(lines) + "\n")
            ref = TextDataset(src, pc)
            speaker_map = json.load(open(os.path.join(pre, "speakers.json")))
            used = {s: speaker_map[s] for s in sorted({l.split("|")[1] for l in lines})}
            items = [ref[i] for i in range(len(ref))]
            batches = list(DataLoader(ref, batch_size=8, collate_fn=ref.collate_fn))
            d.update({f"{ds}_lines": np.array(lines), f"{ds}_speaker_map": json.dumps(used),
                      f"{ds}_cleaners": json.dumps(pc["preprocessing"]["text"]["text_cleaners"]),
                      f"{ds}_phones": np.concatenate([it[2] for it in items]), f"{ds}_phone_lens": np.array([len(it[2]) for it in items]),
                      f"{ds}_ids": np.array([i for b in batches for i in b[0]]), f"{ds}_raw": np.array([r for b in batches for r in b[1]]),
                      f"{ds}_speakers": np.concatenate([b[2] for b in batches]), f"{ds}_texts": np.concatenate([b[3].reshape(-1) for b in batches]),
                      f"{ds}_text_lens": np.concatenate([b[4] for b in batches]), f"{ds}_max_len": np.array([b[5] for b in batches]),
                      f"{ds}_batch_sizes": np.array([len(b[0]) for b in batches])})
            print("frontend", ds, len(lines), "utterances,", len(batches), "batches")
    finally:
        os.chdir(cwd)
    np.savez_compressed(os.path.join(OUT, "frontend_val.npz"), **d)


PARTS = ("base", "pins", "frontend")


def main(parts=PARTS):
    torch.set_num_threads(1)      # pin the thread count: run-to-run bitwise reproducible (SURVEY.md Appendix D)
    FastSpeech2, hifigan = ref_import.load()
    os.makedirs(OUT, exist_ok=True)
    tmp = tempfile.mkdtemp()
    if "pins" in parts:
        gen_pins(FastSpeech2, hifigan, tmp)
    if "frontend" in parts:
        gen_frontend()
    if "base" in parts:
        gen_base(FastSpeech2, hifigan, tmp)


def gen_base(FastSpeech2, hifigan, tmp):
    keys = {}
    cases = [("fs2_lj", "LJSpeech", 11, dict(batch=2, max_len=24, seed=21, min_len=15), dict(p_control=1.0, e_control=1.0, d_control=1.0)),
             ("fs2_libri", "LibriTTS", 12, dict(batch=3, max_len=32, seed=22, min_len=12, n_speakers=904),
              dict(p_control=1.1, e_control=0.9, d_control=0.8))]
    for name, ds, seed, bk, ctl in cases:
        pc, mc = configs.make_configs(ds, tmp)
        sd = synth.fastspeech2_state_dict(pc, mc, seed=seed)
        ref = FastSpeech2(pc, mc)
        ref.load_state_dict(sd, strict=True)
        ref.eval()
        keys[ds] = {k: list(v.shape) for k, v in ref.state_dict().items()}
        spk, texts, lens, L = synth.make_batch(**bk)
        with torch.no_grad():
            out = ref(spk, texts, lens, L, **ctl)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), seed=seed, speakers=spk.numpy(), texts=texts.numpy(),
                            src_lens=lens.numpy(), max_src_len=L, mel=out[0].numpy(), postnet_mel=out[1].numpy(),
                            p_pred=out[2].numpy(), e_pred=out[3].numpy(), logd=out[4].numpy(), d_rounded=out[5].numpy(),
                            src_masks=out[6].numpy(), mel_masks=out[7].numpy(), mel_lens=out[9].numpy(), **ctl)
        print(name, "mel", tuple(out[0].shape), "mel_lens", out[9].tolist())

    h = hifigan.AttrDict(configs.HIFIGAN_CONFIG)
    seed = 13
    hsd = synth.hifigan_state_dict(h, seed=seed)
    gen = hifigan.Generator(h)
    gen.load_state_dict(hsd, strict=True)
    keys["hifigan_weight_norm"] = {k: list(v.shape) for k, v in gen.state_dict().items()}
    gen.eval()
    gen.remove_weight_norm()
    keys["hifigan_folded"] = {k: list(v.shape) for k, v in gen.state_dict().items()}
    mel = synth.make_mel(2, 24, seed=23)
    with torch.no_grad():
        wav = gen(mel)
    np.savez_compressed(os.path.join(OUT, "hifigan.npz"), seed=seed, mel=mel.numpy(), wav=wav.numpy())
    print("hifigan wav", tuple(wav.shape), "peak", float(wav.abs().max()))
    # config/LJSpeech_paper: 4-layer decoder, frame-level unnormalised pitch / energy, log-spaced pitch edges (SURVEY.md section 8 f2)
    pc, mc = configs.make_configs("LJSpeech_paper", tmp)
    seed = 14
    sd = paper_state_dict(pc, mc, seed)
    ref = FastSpeech2(pc, mc)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    keys["LJSpeech_paper"] = {k: list(v.shape) for k, v in ref.state_dict().items()}
    spk, texts, lens, L = synth.make_batch(batch=3, max_len=30, seed=24, min_len=14)
    with torch.no_grad():
        out = ref(spk, texts, lens, L, p_control=1.05)
    np.savez_compressed(os.path.join(OUT, "fs2_lj_paper.npz"), seed=seed, speakers=spk.numpy(), texts=texts.numpy(),
                        src_lens=lens.numpy(), max_src_len=L, mel=out[0].numpy(), postnet_mel=out[1].numpy(),
                        p_pred=out[2].numpy(), e_pred=out[3].numpy(), logd=out[4].numpy(), d_rounded=out[5].numpy(),
                        src_masks=out[6].numpy(), mel_masks=out[7].numpy(), mel_lens=out[9].numpy(), p_control=1.05, e_control=1.0, d_control=1.0)
    nb = torch.bucketize(out[2], sd["variance_adaptor.pitch_bins"]).unique().numel()
    print("fs2_lj_paper mel", tuple(out[0].shape), "mel_lens", out[9].tolist(), "distinct log-spaced pitch buckets", nb)

    # the shipped generator checkpoints (real weights): outputs of the unmodified reference Generator on a synthetic mel
    from oracle import real_ckpt
    for name in ("LJSpeech", "universal"):
        gen = hifigan.Generator(h)
        gen.load_state_dict(real_ckpt.read_reference_checkpoint(name), strict=True)     # utils/model.py:62-66
        gen.eval()
        gen.remove_weight_norm()
        mel = synth.make_mel(2, 96, seed=25)
        with torch.no_grad():
            wav = gen(mel)
        np.savez_compressed(os.path.join(OUT, f"hifigan_real_{name}.npz"), mel=mel.numpy(), wav=wav.numpy())
        print("hifigan real", name, tuple(wav.shape), "peak", float(wav.abs().max()))
    with open(os.path.join(OUT, "state_dict_keys.json"), "w") as f:
        json.dump(keys, f, indent=0, sort_keys=True)


if __name__ == "__main__":
    main(sys.argv[1:] or PARTS)
