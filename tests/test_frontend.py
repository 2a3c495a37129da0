"""Batch-mode front-end (fastspeech2_b200/frontend.py) against the reference's TextDataset + DataLoader + to_device
(dataset.py:149-198, synthesize.py:191-198, utils/tools.py:58-65), and its own host logic (bucketing, sharding, prefetch thread)."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fastspeech2_b200 import frontend  # noqa: E402

VOCAB = {s: i + 1 for i, s in enumerate("AA AE AH B D IY K L M N OW S T sp".split())}


def fake_t2s(text, cleaners):
    assert cleaners == ["english_cleaners"]
    return [VOCAB[s] for s in text.strip("{}").split()]


def make_source(tmp_path, n=37, seed=0, speakers=("spkA", "spkB", "spkC")):
    rng = np.random.default_rng(seed)
    syms = list(VOCAB)
    lines = []
    for i in range(n):
        L = int(rng.integers(1, 40))
        ph = " ".join(rng.choice(syms, size=L))
        lines.append(f"utt{i:03d}|{speakers[i % len(speakers)]}|{{{ph}}}|raw text {i}")
    src = tmp_path / "val.txt"
    src.write_text("\n".join(lines) + "\n", encoding="utf-8")
    pre = tmp_path / "pre"
    pre.mkdir()
    (pre / "speakers.json").write_text(json.dumps({s: j for j, s in enumerate(speakers)}))
    cfg = {"preprocessing": {"text": {"text_cleaners": ["english_cleaners"]}}, "path": {"preprocessed_path": str(pre)}}
    return str(src), cfg, lines


def test_file_order_batches_have_the_reference_layout(tmp_path):
    src, cfg, lines = make_source(tmp_path)
    tb = frontend.TextBatches(src, cfg, batch_size=8, text_to_sequence=fake_t2s)
    batches = list(tb)
    assert len(tb) == len(batches) == 5 and [len(b[0]) for b in batches] == [8, 8, 8, 8, 5]
    k = 0
    for ids, raw, spk, texts, lens, mx in batches:
        assert spk.dtype == np.int64 and texts.dtype == np.int64 and lens.dtype == np.int64 and texts.shape == (len(ids), mx) and mx == lens.max()
        for r in range(len(ids)):
            name, s, t, rw = lines[k].split("|")
            want = fake_t2s(t, ["english_cleaners"])
            assert ids[r] == name and raw[r] == rw and spk[r] == ["spkA", "spkB", "spkC"].index(s)
            assert lens[r] == len(want) and texts[r, : lens[r]].tolist() == want and not texts[r, lens[r]:].any()
            k += 1
    assert k == len(lines)


def test_bucketing_covers_every_utterance_once_and_cuts_padding(tmp_path):
    src, cfg, lines = make_source(tmp_path, n=101, seed=3)
    plain = frontend.TextBatches(src, cfg, batch_size=8, text_to_sequence=fake_t2s)
    buck = frontend.TextBatches(src, cfg, batch_size=8, bucket=True, text_to_sequence=fake_t2s)
    seen = [i for b in buck for i in b[0]]
    assert sorted(seen) == sorted(l.split("|")[0] for l in lines) and len(seen) == len(set(seen))
    maxes = [b[5] for b in buck]
    assert maxes == sorted(maxes, reverse=True)                         # longest first: the first batch sizes the workspaces
    assert buck.padded_fraction() < 0.25 * plain.padded_fraction()


def test_rank_sharding_partitions_whole_batches(tmp_path):
    src, cfg, _ = make_source(tmp_path, n=90)
    whole = [b[0] for b in frontend.TextBatches(src, cfg, batch_size=8, text_to_sequence=fake_t2s)]
    for world in (2, 3, 8):
        parts = [[b[0] for b in frontend.TextBatches(src, cfg, batch_size=8, text_to_sequence=fake_t2s, rank=r, world=world)] for r in range(world)]
        assert [b for p in parts for b in p] == whole                     # same batch composition for every GPU count, contiguous blocks
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_malformed_line_and_unknown_speaker_raise(tmp_path):
    src, cfg, _ = make_source(tmp_path, n=3)
    with open(src, "a", encoding="utf-8") as f:
        f.write("only|three|fields\n")
    with pytest.raises(ValueError, match="4"):
        frontend.TextBatches(src, cfg, text_to_sequence=fake_t2s)
    (tmp_path / "b").mkdir()
    src2, cfg2, _ = make_source(tmp_path / "b", n=3, speakers=("nobody",))
    json.dump({"someone": 0}, open(os.path.join(cfg2["path"]["preprocessed_path"], "speakers.json"), "w"))
    with pytest.raises(KeyError):                                         # the reference's speaker_map lookup raises KeyError too (dataset.py:170)
        list(frontend.TextBatches(src2, cfg2, text_to_sequence=fake_t2s))


def test_prefetch_thread_stops_when_the_consumer_leaves_and_surfaces_errors(tmp_path):
    import threading
    src, cfg, _ = make_source(tmp_path, n=64)
    tb = frontend.TextBatches(src, cfg, batch_size=4, text_to_sequence=fake_t2s, prefetch=1)
    it = iter(tb)
    next(it); it.close()
    for _ in range(50):
        if not any(t.name == "fs2-text-batches" and t.is_alive() for t in threading.enumerate()):
            break
        time.sleep(0.05)
    assert not any(t.name == "fs2-text-batches" and t.is_alive() for t in threading.enumerate())
    tb.collate = lambda idx: (_ for _ in ()).throw(RuntimeError("boom"))
    with pytest.raises(RuntimeError, match="boom"):
        list(tb)


def test_device_batches_on_cpu_equal_to_device(tmp_path):
    import torch
    src, cfg, _ = make_source(tmp_path, n=21)
    tb = frontend.TextBatches(src, cfg, batch_size=8, text_to_sequence=fake_t2s)
    for (ids, raw, spk, texts, lens, mx), (ids2, raw2, s_t, t_t, l_t, mx2) in zip(list(tb), tb.device_batches("cpu")):
        assert ids == ids2 and raw == raw2 and mx == mx2
        assert s_t.dtype == t_t.dtype == l_t.dtype == torch.int64
        assert torch.equal(s_t, torch.from_numpy(spk)) and torch.equal(t_t, torch.from_numpy(texts)) and torch.equal(l_t, torch.from_numpy(lens))


@pytest.mark.gpu
def test_device_batches_on_cuda_stage_through_pinned_slots(tmp_path):
    import torch
    src, cfg, _ = make_source(tmp_path, n=75, seed=5)
    tb = frontend.TextBatches(src, cfg, batch_size=8, bucket=True, text_to_sequence=fake_t2s, prefetch=2)
    host = list(tb)
    got = []
    for ids, raw, s_t, t_t, l_t, mx in tb.device_batches("cuda:0"):
        assert s_t.is_cuda and t_t.is_cuda and l_t.is_cuda
        got.append((ids, raw, (s_t * 1).cpu(), (t_t * 1).cpu(), (l_t * 1).cpu(), mx))      # a kernel on the consumer's stream reads them
    assert len(got) == len(host)
    for (ids, raw, spk, texts, lens, mx), (ids2, raw2, s_t, t_t, l_t, mx2) in zip(host, got):
        assert ids == ids2 and raw == raw2 and mx == mx2
        assert torch.equal(s_t, torch.from_numpy(spk)) and torch.equal(t_t, torch.from_numpy(texts)) and torch.equal(l_t, torch.from_numpy(lens))


def test_against_the_reference_dataloader_on_its_shipped_val_files(tmp_path):
    """Every 8th line of the three `preprocessed_data/*/val.txt` files the reference ships (English ARPAbet and Mandarin pinyin):
    TextBatches / device_batches and OUR TextDataset under a stock DataLoader(batch_size=8), against the batches the reference's own
    TextDataset + DataLoader produced (tests/golden/frontend_val.npz, oracle/gen_golden.py gen_frontend).  Phoneme ids are the
    reference's text_to_sequence output, recorded per utterance."""
    import torch
    from torch.utils.data import DataLoader
    z = np.load(os.path.join(ROOT, "tests", "golden", "frontend_val.npz"))
    n = 0
    for ds_name in ("LJSpeech", "LibriTTS", "AISHELL3"):
        g = lambda k: z[f"{ds_name}_{k}"]
        lines, cleaners = [str(l) for l in g("lines")], json.loads(str(g("cleaners")))
        phones = np.split(g("phones"), np.cumsum(g("phone_lens"))[:-1])
        seq_of = {l.split("|")[2]: p for l, p in zip(lines, phones)}

        def t2s(text, c):
            assert c == cleaners
            return seq_of[text]

        d = tmp_path / ds_name
        d.mkdir()
        (d / "val.txt").write_text("\n".join(lines) + "\n", encoding="utf-8")
        (d / "speakers.json").write_text(str(g("speaker_map")))
        src, pc = str(d / "val.txt"), {"preprocessing": {"text": {"text_cleaners": cleaners}}, "path": {"preprocessed_path": str(d)}}
        sizes, mxs = g("batch_sizes"), g("max_len")
        rows, flat = np.cumsum(np.r_[0, sizes]), np.cumsum(np.r_[0, sizes * mxs])
        want = [(list(g("ids")[rows[b]:rows[b + 1]]), list(g("raw")[rows[b]:rows[b + 1]]), g("speakers")[rows[b]:rows[b + 1]],
                 g("texts")[flat[b]:flat[b + 1]].reshape(sizes[b], mxs[b]), g("text_lens")[rows[b]:rows[b + 1]], mxs[b]) for b in range(len(sizes))]
        ours_ds = frontend.TextDataset(src, pc, text_to_sequence=t2s)
        via_loader = list(DataLoader(ours_ds, batch_size=8, collate_fn=ours_ds.collate_fn))
        tb = frontend.TextBatches(src, pc, batch_size=8, text_to_sequence=t2s)
        direct, dev = list(tb), list(tb.device_batches("cpu"))
        assert len(want) == len(via_loader) == len(direct) == len(dev) == 8
        for w, a, b, dv in zip(want, via_loader, direct, dev):
            for got in (a, b):
                assert got[0] == w[0] and got[1] == w[1] and got[5] == w[5] and type(got[5]) is type(w[5])
                for i in (2, 3, 4):
                    assert got[i].dtype == w[i].dtype and got[i].shape == w[i].shape and np.array_equal(got[i], w[i]), (ds_name, i)
            assert dv[0] == w[0] and dv[1] == w[1] and dv[5] == w[5]
            for i in (2, 3, 4):
                assert dv[i].dtype == torch.int64 and torch.equal(dv[i], torch.from_numpy(w[i]).long())
            n += len(w[0])
        speaker_map = json.loads(str(g("speaker_map")))
        for i, line in enumerate(lines):
            name, spk, _, raw = line.split("|")
            item = ours_ds[i]
            assert item[0] == name and item[1] == speaker_map[spk] and np.array_equal(item[2], phones[i]) and item[3] == raw
    assert n == 192
