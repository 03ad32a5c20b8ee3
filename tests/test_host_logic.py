"""CPU tests of the host side: C-ABI library loads and exports every declared symbol, weight re-layout functions
are exact, the Python surface mirrors the reference's keys / signatures / error behaviour, and compute refuses to
run without a GPU (no CPU fallback)."""
import ctypes
import inspect
import re
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

import gigaam_b200 as gigaam
from gigaam_b200 import _lib, engine, synthetic
from gigaam_b200.decoding import Tokenizer
from gigaam_b200.timestamps_utils import compute_frame_shift, frames_to_words

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "gigaam_b200.h").read_text()
    declared = set(re.findall(r"\b(gam_[a-z0-9_]+)\s*\(", header))
    assert {"gam_create", "gam_logmel", "gam_encode", "gam_ctc_greedy", "gam_rnnt_greedy"} <= declared
    lib = _lib.load()
    for sym in sorted(declared):
        assert hasattr(lib, sym), f"{sym} declared in include/gigaam_b200.h but not exported"
    assert set(_lib.EXPORTS) == declared
    assert lib.gam_version() >= 100
    assert lib.gam_profile_class_count() > 10


def test_struct_layouts_match_header():
    header = (ROOT / "include" / "gigaam_b200.h").read_text()
    layer = header[header.index("typedef struct gam_layer_weights"): header.index("} gam_layer_weights;")]
    names = re.findall(r"[\*\s](\w+)\s*[;,]", re.sub(r"/\*.*?\*/", "", layer, flags=re.S))
    assert tuple(names) == _lib.LAYER_FIELDS
    assert ctypes.sizeof(_lib.GamLayerWeights) == 8 * len(_lib.LAYER_FIELDS)
    cfg = header[header.index("typedef struct gam_config"): header.index("} gam_config;")]
    cfg_names = re.findall(r"(\w+)\s*[;,]", re.sub(r"/\*.*?\*/", "", cfg, flags=re.S))
    assert cfg_names == [n for n, _ in _lib.GamConfig._fields_]


def test_no_cpu_fallback():
    ck = gigaam.synthetic_checkpoint("v2_ctc", n_layers=1)
    model = gigaam.load_model("v2_ctc", device="cpu", checkpoint=ck)
    with pytest.raises(RuntimeError, match="no CPU"):
        model(torch.zeros(1, 16000), torch.tensor([16000]))
    with pytest.raises(RuntimeError, match="CUDA"):
        engine.Engine(ck["cfg"], ck["state_dict"], torch.device("cpu"))


def test_state_dict_keys_and_first_parameter_match_reference_schema():
    for name, cls in [("v2_ctc", gigaam.GigaAMASR), ("v2_rnnt", gigaam.GigaAMASR), ("v2_ssl", gigaam.GigaAM)]:
        ck = gigaam.synthetic_checkpoint(name, n_layers=2)
        model = gigaam.load_model(name, device="cpu", checkpoint=ck)
        assert type(model) is cls
        assert list(model.state_dict().keys()) == list(ck["state_dict"].keys()) or set(model.state_dict()) == set(ck["state_dict"])
        assert next(iter(model.named_parameters()))[0] == "encoder.pre_encode.conv.0.weight"  # -> _dtype / _device
        for k, v in model.state_dict().items():
            assert torch.equal(v, ck["state_dict"][k]), k
    # SURVEY Appendix B spot checks
    sd = gigaam.synthetic_checkpoint("v2_rnnt", n_layers=1)["state_dict"]
    assert sd["encoder.pre_encode.out.weight"].shape == (768, 12288)
    assert sd["encoder.layers.0.conv.pointwise_conv1.weight"].shape == (1536, 768, 1)
    assert sd["head.decoder.lstm.weight_ih_l0"].shape == (1280, 320)
    assert sd["head.joint.joint_net.1.weight"].shape == (34, 320)
    assert sd["preprocessor.featurizer.0.mel_scale.fb"].shape == (201, 64)


def test_load_model_signature_and_errors():
    sig = inspect.signature(gigaam.load_model)
    assert list(sig.parameters)[:5] == ["model_name", "fp16_encoder", "use_flash", "device", "download_root"]
    assert sig.parameters["fp16_encoder"].default is True and sig.parameters["use_flash"].default is False
    with pytest.raises(ValueError, match="not found"):
        gigaam.load_model("v9_ctc", device="cpu")
    with pytest.raises(FileNotFoundError):
        gigaam.load_model("v2_ctc", device="cpu", download_root="/nonexistent")


def test_glu_permutation_and_bn_fold_are_exact():
    d = 768
    perm = engine.glu_row_permutation(d)
    assert sorted(perm.tolist()) == list(range(2 * d))
    g = torch.Generator().manual_seed(0)
    w1 = torch.randn(2 * d, d, generator=g)
    x = torch.randn(5, d, generator=g)
    y = x @ w1[perm].t()                                           # accumulator column order
    t = y.view(5, d // 128, 2, 128)
    glu_tiles = (t[:, :, 0] * torch.sigmoid(t[:, :, 1])).reshape(5, d)
    assert torch.allclose(glu_tiles, F.glu(x @ w1.t(), dim=-1), atol=1e-5)
    # BatchNorm folding == conv -> batch_norm(eval)
    k = 31
    dw, db = torch.randn(d, k, generator=g), torch.randn(d, generator=g)
    gamma, beta = torch.randn(d, generator=g), torch.randn(d, generator=g)
    mean, var = torch.randn(d, generator=g), torch.rand(d, generator=g) + 0.1
    xin = torch.randn(2, d, 40, generator=g)
    ref = F.batch_norm(F.conv1d(xin, dw[:, None], db, padding=15, groups=d), mean, var, gamma, beta, False, 0.0, 1e-5)
    fw, fb = engine.fold_batchnorm(dw, db, gamma, beta, mean, var)
    assert torch.allclose(F.conv1d(xin, fw[:, None], fb, padding=15, groups=d), ref, atol=1e-4)


def test_conv2_and_linear_permutations_reproduce_reference_ops():
    """Implicit-GEMM K order (tap, channel) and the (f, c) flatten order give the reference's conv2d + Linear."""
    g = torch.Generator().manual_seed(1)
    C, F1, T1 = 8, 6, 9
    x = torch.randn(2, C, T1, F1, generator=g)                     # [B, C, T, F] as the reference's conv sees it
    w2 = torch.randn(C, C, 3, 3, generator=g)
    ref = F.conv2d(x, w2, stride=2, padding=1)                     # [B, C, T2, F2]
    T2, F2 = ref.shape[2], ref.shape[3]
    xp = F.pad(x, (1, 1, 1, 1))
    rows = []
    for t2 in range(T2):
        for f2 in range(F2):
            taps = [xp[:, :, 2 * t2 + kt, 2 * f2 + kf] for kt in range(3) for kf in range(3)]   # each [B, C]
            rows.append(torch.cat(taps, dim=1))
    A = torch.stack(rows, 1)                                       # [B, T2*F2, 9C]
    out = A @ engine.pack_conv2_weight(w2).t()
    assert torch.allclose(out.view(2, T2, F2, C).permute(0, 3, 1, 2), ref, atol=1e-4)
    wo = torch.randn(5, C * F2, generator=g)
    y_ref = F.linear(ref.transpose(1, 2).reshape(2, T2, -1), wo)   # reference flatten: index c*F2 + f
    y = out.view(2, T2, F2 * C) @ engine.pack_sub_out_weight(wo, C).t()
    assert torch.allclose(y, y_ref, atol=1e-4)


def test_split_dft_basis_reproduces_rfft_power():
    """[f_hi | f_lo | f_hi] . [d_hi | d_hi | d_lo]^T with the tile row layout == |rfft|^2 (to ~1e-6 relative)."""
    n = 400
    W = engine.split_dft_basis(n).double()                         # [512, 3*448]
    kp = W.shape[1] // 3
    g = torch.Generator().manual_seed(0)
    f = torch.randn(5, n, generator=g).double() * torch.hann_window(n, dtype=torch.float64)
    fp = torch.zeros(5, kp, dtype=torch.float64)
    fp[:, :n] = f * 0.05 * engine.DFT_FRAME_SCALE                 # quiet signal, pre-scaled like frames_split_kernel
    hi = fp.to(torch.float16).double()
    lo = (fp - hi).to(torch.float16).double()
    acc = torch.cat([hi, lo, hi], 1) @ W.t()                       # [5, 512]
    t = acc.view(5, 2, 2, 128)                                     # tile, (cos|sin), bin
    power = (t[:, :, 0] ** 2 + t[:, :, 1] ** 2).reshape(5, 256)[:, : n // 2 + 1]
    power = power / (engine.DFT_FRAME_SCALE * engine.DFT_BASIS_SCALE) ** 2
    f = f * 0.05
    want = torch.fft.rfft(f, dim=-1).abs() ** 2
    assert float(((power - want).abs() / (want.abs() + 1e-6)).max()) < 1e-4
    assert float((power - want).abs().max() / want.abs().max()) < 1e-6


def test_length_arithmetic_matches_reference_formulae():
    from gigaam_b200.encoder import StridingSubsampling
    from gigaam_b200.preprocess import FeatureExtractor
    fe = FeatureExtractor(16000, 64)
    n = torch.tensor([80000, 160000, 240000, 400000, 3200, 5000, 399, 1])
    assert fe.out_len(n).tolist() == [501, 1001, 1501, 2501, 21, 32, 3, 1]
    sub = StridingSubsampling("conv2d", 3)
    assert sub.calc_output_length(fe.out_len(n)).tolist() == [126, 251, 376, 626, 6, 8, 1, 1]
    fe3 = FeatureExtractor(16000, 64, win_length=320, n_fft=320, hop_length=160, center=False)
    assert fe3.out_len(torch.tensor([160000])).tolist() == [999]
    assert StridingSubsampling("conv1d", 5).calc_output_length(torch.tensor([999])).tolist() == [250]


def test_frontend_buffers_match_torchaudio():
    ta = pytest.importorskip("torchaudio")
    ms = ta.transforms.MelSpectrogram(sample_rate=16000, n_mels=64, win_length=400, hop_length=160, n_fft=400)
    assert torch.allclose(synthetic.hann_window(400), ms.spectrogram.window, atol=1e-7)
    assert torch.allclose(synthetic.mel_filterbank(201, 64, 16000), ms.mel_scale.fb, atol=1e-6)


def test_tokenizer_and_word_timestamps():
    tok = Tokenizer(list("ab c"))
    assert len(tok) == 4 and tok.decode([0, 1, 2, 3]) == "ab c" and tok.id_to_str(2) == " "
    words = frames_to_words(tok, [0, 1, 2, 3], [2, 3, 5, 9], compute_frame_shift(16000, 25))
    assert [w.text for w in words] == ["ab", "c"]
    assert words[0].start == pytest.approx(0.08) and words[0].end == pytest.approx(0.16)
    assert words[1].start == pytest.approx(0.36) and words[1].end == pytest.approx(0.40)


def test_synthetic_audio_is_deterministic_and_bounded():
    a, la = synthetic.synthetic_audio(3, 1.0, seed=5, ragged=True)
    b, lb = synthetic.synthetic_audio(3, 1.0, seed=5, ragged=True)
    assert torch.equal(a, b) and torch.equal(la, lb)
    assert a.dtype == torch.float32 and float(a.abs().max()) <= 1.1
    assert la[0] == 16000 and (la[1:] < 16000).all()
    assert float(a[1, int(la[1]):].abs().max()) == 0.0


def test_transcription_result_str():
    r = gigaam.TranscriptionResult(text="привет")
    assert str(r) == "привет" and r.words is None


def test_checkpoint_with_omegaconf_cfg_loads_without_omegaconf(tmp_path):
    """A reference `.ckpt` pickles its cfg as omegaconf objects (gigaam/__init__.py:167).  Build a pickle with the same
    shape from throw-away classes registered under the omegaconf module names, drop those modules, and read it back with
    gigaam_b200.ckpt: plain containers with the values, tensors intact, and `load_model(<path>)`-style use works."""
    import sys
    import types as pytypes
    from gigaam_b200 import ckpt
    if "omegaconf" in sys.modules and not isinstance(sys.modules["omegaconf"], pytypes.ModuleType):
        pytest.skip("unexpected omegaconf module object")
    try:
        import omegaconf  # noqa: F401
        pytest.skip("omegaconf is installed: the ordinary torch.load path is used")
    except ImportError:
        pass
    names = {"omegaconf": [], "omegaconf.base": ["ContainerMetadata", "NodeMetadata"], "omegaconf.dictconfig": ["DictConfig"],
             "omegaconf.listconfig": ["ListConfig"], "omegaconf.nodes": ["AnyNode", "StringNode", "IntegerNode"]}
    mods, cls = {}, {}
    for mod, classes in names.items():
        m = pytypes.ModuleType(mod)
        for c in classes:
            k = type(c, (), {})
            k.__module__ = mod
            setattr(m, c, k)
            cls[c] = k
        mods[mod] = m

    def node(kind, val, parent=None):
        n = cls[kind]()
        n.__dict__.update(_val=val, _parent=parent, _flags_cache=None)
        meta = cls["NodeMetadata"]()
        meta.__dict__.update(ref_type=object, object_type=None, optional=True, key=None, flags=None)
        n.__dict__["_metadata"] = meta
        return n

    def container(kind, content):
        c = cls[kind]()
        meta = cls["ContainerMetadata"]()
        meta.__dict__.update(ref_type=object, object_type=dict, optional=True, key=None, flags={}, key_type=str, element_type=object)
        c.__dict__.update(_metadata=meta, _parent=None, _flags_cache=None, _content=content)
        return c

    enc = container("DictConfig", {"_target_": node("StringNode", "gigaam.encoder.ConformerEncoder"), "n_layers": node("IntegerNode", 16),
                                   "subsampling": node("AnyNode", "conv2d")})
    vocab = container("ListConfig", [node("StringNode", " "), node("StringNode", "а")])
    cfg = container("DictConfig", {"model_name": node("StringNode", "v2_ctc"), "encoder": enc,
                                   "decoding": container("DictConfig", {"vocabulary": vocab})})
    path = tmp_path / "fake.ckpt"
    sys.modules.update(mods)
    try:
        torch.save({"cfg": cfg, "state_dict": {"w": torch.arange(6.0).view(2, 3)}}, path)
    finally:
        for mod in mods:
            sys.modules.pop(mod, None)
    got = ckpt.load_checkpoint(str(path))
    assert got["cfg"] == {"model_name": "v2_ctc",
                          "encoder": {"_target_": "gigaam.encoder.ConformerEncoder", "n_layers": 16, "subsampling": "conv2d"},
                          "decoding": {"vocabulary": [" ", "а"]}}
    assert torch.equal(got["state_dict"]["w"], torch.arange(6.0).view(2, 3))
    assert gigaam._torch_load_ckpt(str(path))["cfg"]["encoder"]["n_layers"] == 16


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the compiled reference of oracle/_ref -- else the oracle port -- timed on the host cores) must print exactly one JSON line on stdout
    with the keys the driver reads, also when launched as a non-zero rank (which stays silent)."""
    import json
    import os
    import subprocess
    import sys
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "utt/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["metric"].startswith("utterances/sec")
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT), env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_rel_pos_weight_packing_reproduces_the_reference_scores():
    """The load-time re-layout of the rel_pos attention (engine.pack_rel_pos_qkv, engine.rel_pos_embedding, pos_proj) in
    fp32 on the CPU: one projection [q+u | q+v | k | v], position rows read from the fixed 2*640-1 table at
    REL_POS_MAX_T-1-(i-j), must give the oracle's RelPositionMultiHeadAttention (gigaam/encoder.py:208-228)."""
    from oracle import gigaam_oracle as orc
    torch.manual_seed(5)
    d, H, T, B = 768, 16, 37, 2
    dk, L = d // H, _lib.REL_POS_MAX_T
    q = "a."
    sd = {q + f"linear_{n}.weight": torch.randn(d, d) / d ** 0.5 for n in ("q", "k", "v", "out", "pos")}
    sd.update({q + f"linear_{n}.bias": torch.randn(d) * 0.1 for n in ("q", "k", "v", "out")})
    sd[q + "pos_bias_u"], sd[q + "pos_bias_v"] = torch.randn(H, dk) * 0.2, torch.randn(H, dk) * 0.2
    x = torch.randn(B, T, d)
    key_valid = torch.arange(T)[None, :] < torch.tensor([T, 20])[:, None]
    want = orc.rel_pos_mhsa(x, sd, q, H, orc.rel_pos_table(T, d), key_valid)
    # the engine's packing
    w4, b4 = engine.pack_rel_pos_qkv(sd[q + "linear_q.weight"], sd[q + "linear_q.bias"], sd[q + "linear_k.weight"], sd[q + "linear_k.bias"],
                                     sd[q + "linear_v.weight"], sd[q + "linear_v.bias"], sd[q + "pos_bias_u"], sd[q + "pos_bias_v"])
    assert w4.shape == (4 * d, d) and b4.shape == (4 * d,)
    pe = engine.rel_pos_embedding(L, d)
    assert pe.shape == (2 * L - 1, d) and torch.equal(pe[L - T: L + T - 1], orc.rel_pos_table(T, d))
    pos_proj = pe @ sd[q + "linear_pos.weight"].t()
    qkv = (x @ w4.t() + b4).view(B, T, 4, H, dk)
    qu, qv, k, v = (qkv[:, :, i].transpose(1, 2) for i in range(4))
    p = pos_proj.view(2 * L - 1, H, dk).transpose(0, 1)                      # [H, 2L-1, dk]
    row = (L - 1) - (torch.arange(T)[:, None] - torch.arange(T)[None, :])     # table row of relative position i - j
    bd = torch.einsum("bhid,hijd->bhij", qv, p[:, row])                        # what the kernel's skewed window MMA computes
    sc = (qu @ k.transpose(-1, -2) + bd) / dk ** 0.5
    sc = sc.masked_fill(~key_valid[:, None, None, :], float("-inf"))
    o = (torch.softmax(sc, -1) @ v).transpose(1, 2).reshape(B, T, d)
    got = F.linear(o, sd[q + "linear_out.weight"], sd[q + "linear_out.bias"])
    valid_q = key_valid
    assert float((got[valid_q] - want[valid_q]).abs().max()) < 2e-4


def test_longform_result_type_and_batch_planning():
    """Host side of transcribe_longform (gigaam/model.py:195-259, gigaam/types.py:38-67): result helpers, length
    bucketing (every segment exactly once, batches bounded, less padding than arrival order) and the energy splitter."""
    from gigaam_b200.longform import padding_waste, plan_batches, split_on_energy
    segs = [gigaam.Segment("a b", 0.0, 1.0, [gigaam.Word("a", 0.1, 0.2), gigaam.Word("b", 0.3, 0.4)]), gigaam.Segment("c", 1.0, 2.0, [])]
    res = gigaam.LongformTranscriptionResult(segments=segs)
    assert str(res) == res.text == "a b c" and len(res) == 2 and [s.text for s in res] == ["a b", "c"]
    assert res.has_word_timestamps and [w.text for w in res.words] == ["a", "b"]
    assert not gigaam.LongformTranscriptionResult(segments=[]).has_word_timestamps
    gen = torch.Generator().manual_seed(3)
    lengths = torch.randint(8000, 352000, (37,), generator=gen).tolist()
    batches = plan_batches(lengths, 8)
    assert sorted(i for b in batches for i in b) == list(range(37)) and max(len(b) for b in batches) == 8 and len(batches) == 5
    arrival = [list(range(i, min(i + 8, 37))) for i in range(0, 37, 8)]
    assert padding_waste(lengths, batches) < 0.5 * padding_waste(lengths, arrival)
    with pytest.raises(ValueError):
        plan_batches(lengths, 0)
    # 60 s: loud / quiet alternation every 10 s -> cuts land inside quiet stretches, every piece <= 22 s, nothing lost
    t = torch.arange(60 * 16000) / 16000.0
    loud = ((t // 10) % 2 == 0).float()
    wav = torch.sin(2 * torch.pi * 220 * t) * (0.5 * loud + 0.001)
    pieces, bounds = split_on_energy(wav)
    assert sum(p.numel() for p in pieces) == wav.numel() and torch.equal(torch.cat(pieces), wav)
    assert all(p.numel() <= 22 * 16000 for p in pieces) and len(pieces) == len(bounds) >= 3
    assert bounds[0][0] == 0.0 and bounds[-1][1] == pytest.approx(60.0)
    for (s0, e0), (s1, _) in zip(bounds, bounds[1:]):
        assert e0 == s1 and loud[int(e0 * 16000)] == 0.0


class _Pieces:
    def __init__(self, pieces):
        self.pieces = pieces

    def __len__(self):
        return len(self.pieces)

    def id_to_str(self, i):
        return self.pieces[i]


def test_word_grouping_restatement_and_flag_table_match_the_reference(golden_dir):
    """gigaam_b200.timestamps_utils.frames_to_words against what the reference's own function returned on 300 random
    hypotheses (tests/golden/word_grouping.json, oracle/make_golden.py), and the per-token flag table the device kernel
    consumes."""
    import json
    from gigaam_b200.timestamps_utils import frames_to_words, token_flag_table
    tok = _Pieces(["▁", "▁ab", "cd", "▁e", "f", "▁ ", "g", "▁hij", "k", " ", "\t", "lm"])
    assert token_flag_table(tok).tolist() == [2 | 4, 2, 0, 2, 0, 2 | 4, 0, 2, 0, 1, 4, 0]
    g = json.loads((golden_dir / "word_grouping.json").read_text())
    assert g["pieces"] == tok.pieces and len(g["cases"]) == 300
    for case in g["cases"]:
        got = [[w.text, w.start, w.end] for w in frames_to_words(tok, case["ids"], case["frames"], g["frame_shift"])]
        assert got == case["words"], case


def test_known_answer_transcripts_when_real_checkpoints_are_present():
    """Opportunistic (SURVEY 8c): the reference's own known answers (tests/test_loading.py:19-21 of the reference) are
    asserted when `~/.cache/gigaam/<model>.ckpt` and `~/.cache/gigaam/example.wav` exist AND a GPU is there; nothing is
    downloadable offline, so on the build / bench boxes this test reports a skip with the reason."""
    import os
    import torch
    cache = os.path.expanduser("~/.cache/gigaam")
    wav = os.path.join(cache, "example.wav")
    known = {
        "asr": "ничьих не требуя похвал счастлив уж я надеждой сладкой что дева с трепетом любви посмотрит может быть украдкой на песни грешные мои у лукоморья дуб зеленый",  # noqa: E501
        "v3_e2e_ctc": "Ничьих, не требуя похвал, счастлив уж я надеждой сладкой, Что дева с трепетом любви посмотрит, может быть украдкой На песни грешные мои. У лукоморья дуб зелёный.",  # noqa: E501
        "v3_e2e_rnnt": "Ничьих не требуя похвал, Счастлив уж я надеждой сладкой, Что дева с трепетом любви Посмотрит, может быть, украдкой На песни грешные мои. У лукоморья дуб зелёный.",  # noqa: E501
    }
    names = [n for n in ("v1_ctc", "v1_rnnt", "v2_ctc", "v2_rnnt", "v3_ctc", "v3_rnnt", "v3_e2e_ctc", "v3_e2e_rnnt")
             if os.path.isfile(os.path.join(cache, n + ".ckpt"))]
    if not names or not os.path.isfile(wav) or not torch.cuda.is_available():
        pytest.skip("no real checkpoint + example.wav under ~/.cache/gigaam (or no GPU): known-answer strings not checkable here")
    import gigaam_b200 as gigaam
    for name in names:
        model = gigaam.load_model(name)
        assert str(model.transcribe(wav)) == known.get(name, known["asr"]), name
