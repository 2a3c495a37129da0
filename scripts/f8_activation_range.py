"""How large are the activations that the vocoder's f16 + f8 layers multiply, on the shipped HiFi-GAN checkpoints?

FS2_TC_VARIANT_F8 splits an activation a into a_hi = fp16(a) and a_lo = a - a_hi; the correction MMA takes E4M3 bytes of a_hi and of
a_lo * 2^12.  E4M3 saturates at 448, so a_hi8 saturates from |a| = 448 and a_lo * 2^12 can from |a| = 256 (fp16 ulp 0.25 there).
Below that the split holds ~2^-16 relative; above it the correction term is clipped.

This runs the fp64 HiFi-GAN forward (the same sequence as oracle/fs2_oracle.py::hifigan_forward) on each shipped generator with the
golden mel of tests/golden/hifigan_real_<name>.npz and records max |in_act(x)| -- the value the kernel splits -- for every conv that
the default Generator policy (f8_mask = 0b11110, fs2_resstack stages included) runs in the f16 + f8 format: the upsample
(ConvTranspose1d) of every stage and both convs of every ResBlock pair.  conv_pre is listed for comparison (three-MMA split by default).

    python scripts/f8_activation_range.py [--out profiles/r03/f8_activation_range.json]

Needs the checkpoints: oracle/_ref/hifigan_generator_<name>.pt (made by __graft_entry__.build()) or the original project's zip.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import fs2_oracle as O, real_ckpt  # noqa: E402

E4M3_MAX = 448.0
LO_SAT = 256.0          # |a| from which a_lo * 2^12 can exceed 448


def record(sd, mel, rates=(8, 8, 2, 2), up_k=(16, 16, 4, 4), rb_k=(3, 7, 11), rb_dil=((1, 3, 5),) * 3):
    sd = {k: v.double() for k, v in O.fold_weight_norm(sd).items()}
    rows = []

    def note(layer, a):
        rows.append({"layer": layer, "max_abs_in": float(a.abs().max()), "f8_default": not layer.startswith("conv_pre")})
        return a

    nk = len(rb_k)
    with torch.no_grad():
        x = F.conv1d(note("conv_pre", mel.double()), sd["conv_pre.weight"], sd["conv_pre.bias"], padding=3)
        for i, (u, k) in enumerate(zip(rates, up_k)):
            x = note(f"ups.{i}", F.leaky_relu(x, 0.1))
            x = F.conv_transpose1d(x, sd[f"ups.{i}.weight"], sd[f"ups.{i}.bias"], stride=u, padding=(k - u) // 2)
            acc = None
            for j, (kk, dils) in enumerate(zip(rb_k, rb_dil)):
                r, p = x, f"resblocks.{i * nk + j}"
                for m, d in enumerate(dils):
                    t = F.conv1d(note(f"{p}.convs1.{m}", F.leaky_relu(r, 0.1)), sd[f"{p}.convs1.{m}.weight"], sd[f"{p}.convs1.{m}.bias"],
                                 dilation=d, padding=(kk * d - d) // 2)
                    t = F.conv1d(note(f"{p}.convs2.{m}", F.leaky_relu(t, 0.1)), sd[f"{p}.convs2.{m}.weight"], sd[f"{p}.convs2.{m}.bias"],
                                 padding=(kk - 1) // 2)
                    r = t + r
                acc = r if acc is None else acc + r
            x = acc / nk
        x = F.conv1d(F.leaky_relu(x), sd["conv_post.weight"], sd["conv_post.bias"], padding=3)
    return rows, torch.tanh(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "f8_activation_range.json"))
    args = ap.parse_args()
    result = {"what": "max |in_act(x)| entering each vocoder conv (fp64 forward of the shipped checkpoint on its golden mel)",
              "e4m3_saturation": {"a_hi": E4M3_MAX, "a_lo_times_4096_from": LO_SAT}, "checkpoints": {}}
    for name in ("LJSpeech", "universal"):
        sd = real_ckpt.load(name)
        if sd is None and os.path.exists(real_ckpt.source_zip(name)):
            sd = real_ckpt.read_reference_checkpoint(name)
        if sd is None:
            raise SystemExit(f"checkpoint {name} not available")
        z = np.load(os.path.join(ROOT, "tests", "golden", f"hifigan_real_{name}.npz"))
        rows, wav = record(sd, torch.from_numpy(z["mel"]))
        err = (wav - torch.from_numpy(z["wav"]).double()).abs().max().item()
        assert err < 2e-6, err                    # the recorded forward is the reference's
        f8 = [r for r in rows if r["f8_default"]]
        peak = max(f8, key=lambda r: r["max_abs_in"])
        result["checkpoints"][name] = {"mel_shape": list(z["mel"].shape), "wav_vs_golden": err, "f8_peak": peak,
                                       "f8_layers_within_2x_of_256": [r["layer"] for r in f8 if r["max_abs_in"] >= LO_SAT / 2],
                                       "layers": rows}
        print(f"{name}: {len(f8)} f8 layers, peak {peak['max_abs_in']:.3g} at {peak['layer']}; "
              f">= 128: {result['checkpoints'][name]['f8_layers_within_2x_of_256']}")
        for r in rows:
            print(f"  {r['layer']:<22} {'f8' if r['f8_default'] else '  '} {r['max_abs_in']:10.4g}")
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
