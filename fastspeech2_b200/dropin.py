"""Make the reference's `import model` / `import hifigan` resolve to the B200-native drop-ins.

    import fastspeech2_b200.dropin as dropin; dropin.install()           # programmatic
    python -m fastspeech2_b200.dropin synthesize.py --text ... -p ... -m ... -t ...   # run the untouched reference CLI

`utils/model.py:7-8` does `import hifigan` and `from model import FastSpeech2, ScheduledOptim`; both names are bound here
to `fastspeech2_b200.hifigan` / `fastspeech2_b200.model`, whose classes keep the reference's constructor arguments,
state_dict keys, forward signatures and return values (see INTEGRATION.md).
"""
from __future__ import annotations

import os
import runpy
import sys


def install(force: bool = False) -> None:
    import fastspeech2_b200.hifigan as b_hifigan
    import fastspeech2_b200.model as b_model
    for name, mod in (("model", b_model), ("hifigan", b_hifigan)):
        cur = sys.modules.get(name)
        if cur is not None and cur is not mod and not force:
            raise RuntimeError(f"module {name!r} is already imported from {getattr(cur, '__file__', '?')}; call install() first")
        sys.modules[name] = mod


_pinned = {}


def vocoder_infer(mels, vocoder, model_config, preprocess_config, lengths=None):
    """Drop-in for the reference's `utils.model.vocoder_infer` (utils/model.py:74-92), same arguments and return value (a list of
    int16 numpy arrays, one per utterance, trimmed to `lengths[i]` samples).  The reference copies the fp32 waveform to the host
    and converts / trims there; here `x max_wav_value -> int16` and the trim run on the device (fs2_wav_to_int16), so 2 bytes per
    sample cross PCIe, into pinned memory, asynchronously on the compute stream.  The conversion is numpy's: out-of-range samples wrap
    (a waveform sample of exactly 1.0 becomes -32768) and NaN / inf become 0, so the int16 samples equal the reference's."""
    import torch

    from . import ops
    if model_config["vocoder"]["model"] != "HiFi-GAN":
        raise NotImplementedError("the B200-native path serves the vendored HiFi-GAN vocoder only (MelGAN needs a network fetch upstream)")
    with torch.no_grad():
        wav = vocoder(mels)                                    # [B, 1, N] fp32 on the device
    scale = float(preprocess_config["preprocessing"]["audio"]["max_wav_value"])
    B, _, N = wav.shape
    lens_d = None if lengths is None else torch.as_tensor(lengths).to(wav.device)
    i16 = ops.wav_to_int16(wav[:, 0], lens_d, scale)
    key = (B, N)
    host = _pinned.get(key)
    if host is None:
        host = _pinned[key] = torch.empty(B, N, dtype=torch.int16).pin_memory()
    host.copy_(i16, non_blocking=True)
    lens_h = None if lengths is None else [int(v) for v in torch.as_tensor(lengths).cpu().tolist()]   # syncs after the copy was enqueued
    torch.cuda.current_stream(wav.device).synchronize()
    arr = host.numpy()
    return [arr[i, : (N if lens_h is None else lens_h[i])].copy() for i in range(B)]


def patch_vocoder_infer() -> bool:
    """Rebind `utils.model.vocoder_infer` of the (already importable) reference tree to the device-side version; `utils.tools.synth_samples`
    looks the name up at call time (utils/tools.py:200), so the shipped CLI picks it up unchanged."""
    try:
        import utils.model as um
    except Exception:
        return False
    um.vocoder_infer = vocoder_infer
    return True


def patch_text_dataset() -> bool:
    """Bind `dataset.TextDataset` of the (importable) reference tree to `fastspeech2_b200.frontend.TextDataset`: `synthesize.py` imports the
    name at start-up (synthesize.py:12) and hands the instance and its `collate_fn` to a stock `DataLoader` (synthesize.py:193-198)."""
    try:
        import dataset as ref_dataset
    except Exception:
        return False
    from .frontend import TextDataset
    ref_dataset.TextDataset = TextDataset
    return True


def main(argv=None) -> None:
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        raise SystemExit("usage: python -m fastspeech2_b200.dropin <reference script, e.g. synthesize.py> [script args...]")
    script = os.path.abspath(argv[0])
    install()
    sys.argv = [script] + argv[1:]
    sys.path.insert(0, os.path.dirname(script))       # the reference resolves `utils`, `text`, `dataset` relative to itself
    patch_vocoder_infer()
    patch_text_dataset()
    runpy.run_path(script, run_name="__main__")


if __name__ == "__main__":
    main()
