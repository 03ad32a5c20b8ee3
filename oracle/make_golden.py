"""Generate the fixtures under tests/golden/ from the REAL reference (run where the reference package is readable,
oracle/ref_loader.py) and pin oracle/gigaam_oracle.py against it.

    python oracle/make_golden.py            # writes fixtures, asserts oracle == reference
    python oracle/make_golden.py ragged_v1_ctc word_grouping   # only the named cases

The reference cannot be imported as a package offline (hydra / omegaconf / soundfile are absent,
gigaam/model.py:3-4, gigaam/utils.py:9), so those three are stubbed and its hot-path classes are built
directly from kwargs: gigaam.preprocess.FeatureExtractor, gigaam.encoder.ConformerEncoder,
gigaam.decoder.CTCHead / RNNTHead, gigaam.decoding.CTCGreedyDecoding / RNNTGreedyDecoding.
"""
from __future__ import annotations

import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


from oracle.ref_loader import build_reference  # noqa: E402


def run_case(model_name: str, batch: int, seconds: float, ragged: bool, out_name: str, seed: int = 0):
    from gigaam_b200 import synthetic
    from oracle import gigaam_oracle as orc

    ck = synthetic.synthetic_checkpoint(model_name, seed=seed)
    cfg, sd = ck["cfg"], ck["state_dict"]
    wav, wav_len = synthetic.synthetic_audio(batch, seconds, seed=1234, ragged=ragged)
    root, decoding = build_reference(cfg, sd)
    with torch.inference_mode():
        mel_ref, mel_len_ref = root.preprocessor(wav, wav_len)
        enc_ref, enc_len_ref = root.encoder(mel_ref, mel_len_ref)        # GigaAM.forward on CPU (model.py:33-35)
        pre_ref, _ = root.encoder.pre_encode(x=mel_ref.transpose(1, 2), lengths=mel_len_ref)
        dec_ref = decoding.decode(root.head, enc_ref, enc_len_ref) if decoding is not None else None
        # ---- oracle restatement on the same inputs
        mel_o = orc.log_mel(wav, sd, cfg["preprocessor"])
        pre = cfg["preprocessor"]
        mel_len_o = orc.logmel_out_len(wav_len, pre.get("hop_length", 160), pre.get("win_length", 400), pre.get("center", True))
        enc_o, enc_len_o, stages = orc.encoder_forward(mel_o, mel_len_o, sd, cfg["encoder"], return_all=True)
    valid = (torch.arange(enc_ref.shape[2])[None, :] < enc_len_ref[:, None])

    def rel(a, b):
        return float((a - b).norm() / b.norm())

    report = {
        "mel_max_abs": float((mel_o - mel_ref).abs().max()),
        "mel_len_equal": bool(torch.equal(mel_len_o, mel_len_ref)),
        "pre_encode_rel": rel(stages[0][valid], pre_ref[valid]),
        "enc_rel_valid": rel(enc_o.transpose(1, 2)[valid], enc_ref.transpose(1, 2)[valid]),
        "enc_len_equal": bool(torch.equal(enc_len_o, enc_len_ref)),
    }
    assert report["mel_len_equal"] and report["enc_len_equal"], report
    assert report["mel_max_abs"] < 2e-3, report
    assert report["enc_rel_valid"] < 1e-4, report
    arrays = dict(
        wav_seed=np.int64(1234), batch=np.int64(batch), seconds=np.float64(seconds), ragged=np.bool_(ragged),
        weight_seed=np.int64(seed),
        wav_len=wav_len.numpy(), mel=mel_ref.numpy().astype(np.float32), mel_len=mel_len_ref.numpy(),
        pre_encode=pre_ref.numpy().astype(np.float32),
        enc=enc_ref.numpy().astype(np.float32), enc_len=enc_len_ref.numpy(),
    )
    if dec_ref is not None:
        head = cfg["head"]["type"]
        dec_o = orc.ctc_greedy(enc_ref, enc_len_ref, sd) if head == "ctc" else orc.rnnt_greedy(
            enc_ref, enc_len_ref, sd, cfg["decoding"]["max_symbols_per_step"])
        for b, (text, ids, frames) in enumerate(dec_ref):
            assert ids == dec_o[b][0] and frames == dec_o[b][1], (model_name, b, "oracle decode != reference decode")
            arrays[f"ids_{b}"] = np.asarray(ids, dtype=np.int64)
            arrays[f"frames_{b}"] = np.asarray(frames, dtype=np.int64)
        report["tokens"] = [len(d[1]) for d in dec_ref]
        report["tokens_per_frame"] = float(sum(report["tokens"]) / max(int(enc_len_ref.sum()), 1))
        if head == "ctc":
            lg = orc.ctc_logits(enc_ref, sd)
            top2 = lg.topk(2, dim=-1).values
            arrays["ctc_margin"] = (top2[..., 0] - top2[..., 1]).numpy().astype(np.float32)
    out = ROOT / "tests" / "golden" / out_name
    np.savez_compressed(out, **arrays)
    print(out_name, report, f"{out.stat().st_size / 1024:.0f} KiB")
    return report


RAGGED_SECONDS = [4.0, 0.06, 1.3, 3.1, 0.5, 4.0]   # one 4 s buffer, utterances from full length down to two encoder frames
RAGGED_CHANNELS = 32                               # encoder channels kept per valid frame (a seeded sample of the 768)


def run_ragged_case(model_name: str):
    """The reference's encoder lengths and output on a strongly ragged batch (3 layers deep).  Every valid frame is kept,
    for a fixed sample of the channels, so that the file stays small while a masking or length error still shows."""
    from gigaam_b200 import synthetic
    from oracle import gigaam_oracle as orc

    ck = synthetic.synthetic_checkpoint(model_name, seed=0, n_layers=3)
    root, _ = build_reference(ck["cfg"], ck["state_dict"])
    wav, _ = synthetic.synthetic_audio(len(RAGGED_SECONDS), 4.0, seed=4321)
    wav_len = torch.tensor([int(s * 16000) for s in RAGGED_SECONDS])
    for b, n in enumerate(wav_len.tolist()):
        wav[b, n:] = 0.0
    with torch.inference_mode():
        mel, mel_len = root.preprocessor(wav, wav_len)
        enc, enc_len = root.encoder(mel, mel_len)
        enc_o, enc_len_o = orc.model_forward(wav, wav_len, ck["state_dict"], ck["cfg"])
    assert torch.equal(enc_len.long(), enc_len_o.long()), (enc_len, enc_len_o)
    channels = np.sort(np.random.default_rng(0).choice(enc.shape[1], RAGGED_CHANNELS, replace=False))
    ch = torch.from_numpy(channels)
    enc_valid = torch.cat([enc[b][ch, :n].t() for b, n in enumerate(enc_len.tolist())])     # [sum(enc_len), channels]
    out = ROOT / "tests" / "golden" / f"ragged_{model_name}_l3.npz"
    np.savez_compressed(out, wav_len=wav_len.numpy(), enc_len=enc_len.numpy(), channels=channels,
                        enc_valid=enc_valid.numpy().astype(np.float32))
    print(out.name, enc_len.tolist(), f"{out.stat().st_size / 1024:.0f} KiB")


WORD_PIECES = ["▁", "▁ab", "cd", "▁e", "f", "▁ ", "g", "▁hij", "k", " ", "\t", "lm"]


def run_word_grouping_case():
    """The reference's frames_to_words on 300 random hypotheses over a small SentencePiece-like vocabulary: leading,
    trailing and repeated delimiters, bare U+2581 pieces, whitespace-only pieces, empty hypotheses."""
    import json
    import random
    from oracle.ref_loader import import_reference
    import_reference()
    import gigaam.timestamps_utils as ref_ts

    class Pieces:
        def __len__(self):
            return len(WORD_PIECES)

        def id_to_str(self, i):
            return WORD_PIECES[i]

    rng = random.Random(0)
    cases = []
    for _ in range(300):
        n = rng.randint(0, 40)
        ids = [rng.randrange(len(WORD_PIECES)) for _ in range(n)]
        frames = sorted(rng.randrange(300) for _ in range(n))
        words = [[w.text, w.start, w.end] for w in ref_ts.frames_to_words(Pieces(), ids, frames, 0.04)]
        cases.append({"ids": ids, "frames": frames, "words": words})
    out = ROOT / "tests" / "golden" / "word_grouping.json"
    out.write_text(json.dumps({"pieces": WORD_PIECES, "frame_shift": 0.04, "cases": cases}, separators=(",", ":")) + "\n")
    print(out.name, f"{out.stat().st_size / 1024:.0f} KiB")


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count() or 8)
    cases = {
        "v2_ctc": dict(batch=2, seconds=2.0, ragged=True, out_name="v2_ctc_b2_2s.npz"),
        "v2_rnnt": dict(batch=2, seconds=2.0, ragged=True, out_name="v2_rnnt_b2_2s.npz"),
        # v3 shape (RECALLED, SURVEY App. C): conv1d k5 subsampling, LayerNorm conv-norm, depthwise k5, n_fft 320, center=False
        "v3_e2e_rnnt": dict(batch=2, seconds=2.0, ragged=True, out_name="v3_e2e_rnnt_b2_2s.npz"),
        # v1 shape: the rel_pos attention branch (encoder.py:191-228, 307-334); 6 s so that T' = 151 spans two key blocks
        "v1_ctc": dict(batch=2, seconds=6.0, ragged=True, out_name="v1_ctc_b2_6s.npz"),
    }
    extra = {f"ragged_{m}": (lambda m=m: run_ragged_case(m)) for m in ("v2_ctc", "v3_e2e_rnnt", "v1_ctc")}
    extra["word_grouping"] = run_word_grouping_case
    for name in (sys.argv[1:] or list(cases) + list(extra)):
        if name in extra:
            extra[name]()
        else:
            run_case(name, **cases[name])
