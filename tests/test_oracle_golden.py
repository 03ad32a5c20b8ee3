"""The CPU oracle (oracle/gigaam_oracle.py) against golden vectors produced by the REAL reference modules
(oracle/make_golden.py, run where /root/reference exists).  This is what pins the oracle; the reference itself
cannot travel to the GPU box."""
import numpy as np
import pytest
import torch

from gigaam_b200 import synthetic
from oracle import gigaam_oracle as orc


def _inputs(g):
    wav, wav_len = synthetic.synthetic_audio(int(g["batch"]), float(g["seconds"]), seed=int(g["wav_seed"]), ragged=bool(g["ragged"]))
    assert np.array_equal(wav_len.numpy(), g["wav_len"])
    return wav, wav_len


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.fixture(scope="module")
def ctc_case(golden_dir, v2_ctc_ckpt):
    g = np.load(golden_dir / "v2_ctc_b2_2s.npz")
    wav, wav_len = _inputs(g)
    cfg, sd = v2_ctc_ckpt["cfg"], v2_ctc_ckpt["state_dict"]
    with torch.inference_mode():
        mel = orc.log_mel(wav, sd, cfg["preprocessor"])
        mel_len = orc.logmel_out_len(wav_len, 160, 400, True)
        enc, enc_len, stages = orc.encoder_forward(mel, mel_len, sd, cfg["encoder"], return_all=True)
    return g, cfg, sd, mel, mel_len, enc, enc_len, stages


def test_logmel_matches_reference(ctc_case):
    g, _, _, mel, mel_len, *_ = ctc_case
    assert np.array_equal(mel_len.numpy(), g["mel_len"])
    assert float((mel - torch.from_numpy(g["mel"])).abs().max()) < 1e-4


def test_pre_encode_and_encoder_match_reference(ctc_case):
    g, _, _, _, _, enc, enc_len, stages = ctc_case
    assert np.array_equal(enc_len.numpy(), g["enc_len"])
    valid = torch.arange(enc.shape[2])[None, :] < enc_len[:, None]
    assert _rel(stages[0][valid], torch.from_numpy(g["pre_encode"])[valid]) < 1e-5
    assert _rel(enc.transpose(1, 2)[valid], torch.from_numpy(g["enc"]).transpose(1, 2)[valid]) < 1e-5


def test_ctc_greedy_matches_reference(ctc_case):
    g, _, sd, *_ = ctc_case
    hyp = orc.ctc_greedy(torch.from_numpy(g["enc"]), torch.from_numpy(g["enc_len"]), sd)
    for b, (ids, frames) in enumerate(hyp):
        assert ids == g[f"ids_{b}"].tolist()
        assert frames == g[f"frames_{b}"].tolist()


def test_rnnt_greedy_matches_reference(golden_dir, v2_rnnt_ckpt):
    g = np.load(golden_dir / "v2_rnnt_b2_2s.npz")
    hyp = orc.rnnt_greedy(torch.from_numpy(g["enc"]), torch.from_numpy(g["enc_len"]), v2_rnnt_ckpt["state_dict"], 10)
    total = 0
    for b, (ids, frames) in enumerate(hyp):
        assert ids == g[f"ids_{b}"].tolist()
        assert frames == g[f"frames_{b}"].tolist()
        total += len(ids)
    assert total > 0  # the calibrated blank bias must leave a non-degenerate hypothesis


def test_rel_pos_encoder_matches_reference(golden_dir, v1_ctc_ckpt):
    """v1 shape: the oracle's explicit-index rel_shift against the reference's pad/view one (encoder.py:202-228),
    full 16-layer stack on the reference's own log-mel against its encoder output."""
    g = np.load(golden_dir / "v1_ctc_b2_6s.npz")
    cfg, sd = v1_ctc_ckpt["cfg"], v1_ctc_ckpt["state_dict"]
    assert cfg["encoder"]["self_attention_model"] == "rel_pos"
    with torch.inference_mode():
        enc, enc_len = orc.encoder_forward(torch.from_numpy(g["mel"]), torch.from_numpy(g["mel_len"]), sd, cfg["encoder"])
    assert np.array_equal(enc_len.numpy(), g["enc_len"])
    valid = torch.arange(enc.shape[2])[None, :] < enc_len[:, None]
    assert _rel(enc.transpose(1, 2)[valid], torch.from_numpy(g["enc"]).transpose(1, 2)[valid]) < 1e-5
    hyp = orc.ctc_greedy(torch.from_numpy(g["enc"]), torch.from_numpy(g["enc_len"]), sd)
    for b, (ids, frames) in enumerate(hyp):
        assert ids == g[f"ids_{b}"].tolist() and frames == g[f"frames_{b}"].tolist()


def test_rel_shift_index_matches_pad_view_trick():
    """The reference's rel_shift (pad one column, view as [2T, T], drop the first row) equals reading column
    T-1-i+j of row i -- the index the CUDA kernel skews its position scores by."""
    t = 7
    x = torch.arange(2 * 3 * t * (2 * t - 1), dtype=torch.float32).view(2, 3, t, 2 * t - 1)
    y = torch.nn.functional.pad(x, pad=(1, 0)).view(2, 3, -1, t)[:, :, 1:].view(2, 3, t, 2 * t - 1)[..., :t]
    idx = (t - 1) - torch.arange(t)[:, None] + torch.arange(t)[None, :]
    assert torch.equal(y, torch.gather(x, 3, idx.expand(2, 3, t, t)))


def test_ctc_collapse_edge_cases(v2_ctc_ckpt):
    """Empty lengths, length 1, repeated labels, all blanks (gigaam/decoding.py:76-91 semantics)."""
    sd = v2_ctc_ckpt["state_dict"]
    V1 = sd["head.decoder_layers.0.bias"].numel()
    W = sd["head.decoder_layers.0.weight"].reshape(V1, -1)
    # craft encoder rows that make the head emit chosen labels: e = pinv(W) one-hot * big
    pinv = torch.linalg.pinv(W)
    labels = torch.tensor([[3, 3, V1 - 1, 3, 5, 5, 5, V1 - 1], [V1 - 1] * 8, [1, 2, 3, 4, 5, 6, 7, 8]])
    onehot = torch.nn.functional.one_hot(labels, V1).float() * 50.0
    enc = (onehot @ pinv.t()).transpose(1, 2)                      # [B, d, T]
    got = orc.ctc_greedy(enc, torch.tensor([8, 8, 0]), sd)
    assert got[0] == ([3, 3, 5], [0, 3, 4])
    assert got[1] == ([], [])
    assert got[2] == ([], [])
    got = orc.ctc_greedy(enc, torch.tensor([1, 1, 3]), sd)
    assert got[0] == ([3], [0]) and got[2] == ([1, 2, 3], [0, 1, 2])


def test_compiled_reference_archive_reproduces_the_golden_vectors(golden_dir, v2_ctc_ckpt, monkeypatch):
    """oracle/_ref/gigaam_ref.zip (oracle/build_ref.py: the reference's own modules, byte-compiled; what `bench.py --impl
    reference` times on the GPU box) imported on its own -- not from /root/reference -- gives bit-identical log-mel,
    encoder output and hypotheses to the committed fixtures.  Skipped only where the archive has not been built."""
    from oracle import ref_loader
    if not ref_loader.ARCHIVE.is_file():
        pytest.skip("oracle/_ref/gigaam_ref.zip not built (oracle/build_ref.py needs /root/reference)")
    import subprocess
    import sys
    code = (
        "import sys, numpy as np, torch\n"
        f"sys.path.insert(0, {str(ref_loader.ROOT)!r})\n"
        "from oracle.ref_loader import build_reference, reference_root\n"
        "from gigaam_b200 import synthetic\n"
        "assert reference_root().endswith('gigaam_ref.zip')\n"
        f"g = np.load({str(golden_dir / 'v2_ctc_b2_2s.npz')!r})\n"
        "ck = synthetic.synthetic_checkpoint('v2_ctc', seed=0)\n"
        "root, dec = build_reference(ck['cfg'], ck['state_dict'])\n"
        "wav, wl = synthetic.synthetic_audio(2, 2.0, seed=1234, ragged=True)\n"
        "with torch.inference_mode():\n"
        "    mel, ml = root.preprocessor(wav, wl); enc, el = root.encoder(mel, ml); hyp = dec.decode(root.head, enc, el)\n"
        "assert float((mel - torch.from_numpy(g['mel'])).abs().max()) == 0.0\n"
        "assert float((enc - torch.from_numpy(g['enc'])).abs().max()) == 0.0\n"
        "assert all(list(h[1]) == g[f'ids_{b}'].tolist() and list(h[2]) == g[f'frames_{b}'].tolist() for b, h in enumerate(hyp))\n"
        "print('archive ok')\n")
    env = dict(**__import__("os").environ, GIGAAM_REFERENCE_ARCHIVE_ONLY="1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0 and "archive ok" in res.stdout, res.stderr[-2000:]


@pytest.mark.parametrize("which", ["v2_ctc", "v3_e2e_rnnt", "v1_ctc"])
def test_oracle_matches_the_reference_on_a_strongly_ragged_batch(golden_dir, which):
    """The varlen GPU tests (tests/test_gpu_parity.py::test_varlen_ragged_batch_against_oracle) compare packed-row execution with
    the ORACLE on batches that run from a full buffer down to a two-frame utterance; the other goldens only reach 0.5 of the
    buffer.  This pins the oracle's masking / length arithmetic on such a batch to the reference itself
    (tests/golden/ragged_<model>_l3.npz, oracle/make_golden.py): encoded lengths and the encoder output on every valid frame
    (a fixed sample of 32 channels), for the three encoder shapes (conv2d + BatchNorm + rotary, conv1d + LayerNorm, rel_pos),
    three layers deep."""
    g = np.load(golden_dir / f"ragged_{which}_l3.npz")
    ck = synthetic.synthetic_checkpoint(which, seed=0, n_layers=3)
    secs = [4.0, 0.06, 1.3, 3.1, 0.5, 4.0]
    wav, _ = synthetic.synthetic_audio(len(secs), 4.0, seed=4321)
    wl = torch.tensor([int(s * 16000) for s in secs])
    assert np.array_equal(wl.numpy(), g["wav_len"])
    for b, n in enumerate(wl.tolist()):
        wav[b, n:] = 0.0
    with torch.inference_mode():
        enc_o, el_o = orc.model_forward(wav, wl, ck["state_dict"], ck["cfg"])
    el = torch.from_numpy(g["enc_len"])
    assert torch.equal(el.long(), el_o.long()), (el, el_o)
    assert int(el.min()) <= 2 and int(el.max()) >= 100
    ch = torch.from_numpy(g["channels"])
    a = [enc_o[i][ch, :n].t() for i, n in enumerate(el.tolist())]          # per utterance: [valid frames, channels]
    b = torch.from_numpy(g["enc_valid"]).split(el.tolist())
    rel = _rel(torch.cat(a), torch.cat(b))
    worst = max(_rel(x, y) for x, y in zip(a, b))
    assert rel < 1e-5 and worst < 1e-4, (rel, worst)
