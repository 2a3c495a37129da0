"""The reference converts its waveform with numpy: `(wavs.cpu().numpy() * max_wav_value).astype("int16")` (utils/model.py:82-85).
fs2_wav_to_int16 reproduces that cast -- truncate to int32, keep the low 16 bits; NaN, inf and values outside int32 become 0 -- so that the
drop-in vocoder_infer returns the reference's samples, including for a waveform sample of exactly 1.0.  This pins numpy's side of that
contract: if a numpy release changes the cast, the expected values here (and in tests/test_gpu_ops_ranges.py) change visibly."""
import numpy as np


def test_numpy_float32_to_int16_cast_wraps():
    wav = np.array([1.0, 2.0, 70000 / 32768, np.nan, np.inf, -1.0, -np.inf, 65537 / 32768, 1e5, np.nextafter(np.float32(1), np.float32(0))],
                   np.float32)
    with np.errstate(invalid="ignore"):
        got = (wav * 32768.0).astype("int16")
    assert (wav * 32768.0).dtype == np.float32
    assert got.tolist() == [-32768, 0, 4464, 0, 0, -32768, 0, 1, 0, 32767]
