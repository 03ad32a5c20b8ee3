"""Import the REAL reference modules (test infrastructure; never imported by gigaam_b200/).

Order of preference: /root/reference (the build container), else the byte-compiled archive oracle/_ref/gigaam_ref.zip
(oracle/build_ref.py; the only form in which the reference reaches the GPU box).  GIGAAM_REFERENCE_ARCHIVE_ONLY=1 forces
the archive (used by the CPU test that proves the archive is importable).  hydra / omegaconf / soundfile are absent offline
(gigaam/model.py:3-4, gigaam/utils.py:9) and are stubbed; the hot-path classes are then built directly from kwargs:
gigaam.preprocess.FeatureExtractor, gigaam.encoder.ConformerEncoder, gigaam.decoder.CTCHead / RNNTHead,
gigaam.decoding.CTCGreedyDecoding / RNNTGreedyDecoding.
"""
from __future__ import annotations

import os
import sys
import types
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]


ARCHIVE = ROOT / "oracle" / "_ref" / "gigaam_ref.zip"


def reference_root() -> str | None:
    """sys.path entry that provides the reference's `gigaam` package, or None."""
    if os.environ.get("GIGAAM_REFERENCE_ARCHIVE_ONLY", "0") != "1":
        for cand in (os.environ.get("GIGAAM_REFERENCE"), "/root/reference"):
            try:
                if cand and (Path(cand) / "gigaam" / "encoder.py").is_file():
                    return cand
            except OSError:  # not readable by this user: try the next candidate
                pass
    return str(ARCHIVE) if ARCHIVE.is_file() else None


def import_reference():
    """-> (preprocess, encoder, decoder, decoding) modules of the reference, or raises ImportError."""
    root = reference_root()
    if root is None:
        raise ImportError("the reference is neither at /root/reference nor compiled into oracle/_ref (run oracle/build_ref.py)")
    for name in ("hydra", "hydra.utils", "omegaconf", "soundfile"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["hydra"].utils = sys.modules["hydra.utils"]
    sys.modules["omegaconf"].DictConfig = dict
    sys.modules["omegaconf"].ListConfig = list
    if root not in sys.path:
        sys.path.insert(0, root)
    import gigaam.decoder as ref_decoder
    import gigaam.decoding as ref_decoding
    import gigaam.encoder as ref_encoder
    import gigaam.preprocess as ref_preprocess
    return ref_preprocess, ref_encoder, ref_decoder, ref_decoding


def build_reference(cfg, sd):
    """Instantiate the reference modules for a plain-dict cfg and load the seeded state_dict (strict).
    -> (root nn.Module with .preprocessor / .encoder / .head, decoding object or None)"""
    rp, re_, rd, rdec = import_reference()
    mods = {"preprocessor": rp.FeatureExtractor(**dict(cfg["preprocessor"])), "encoder": re_.ConformerEncoder(**cfg["encoder"])}
    head = cfg.get("head")
    decoding = None
    if head is not None:
        if head["type"] == "ctc":
            mods["head"] = rd.CTCHead(head["feat_in"], head["num_classes"])
            decoding = rdec.CTCGreedyDecoding(cfg["decoding"]["vocabulary"])
        else:
            mods["head"] = rd.RNNTHead(head["decoder"], head["joint"])
            decoding = rdec.RNNTGreedyDecoding(cfg["decoding"]["vocabulary"], None, cfg["decoding"]["max_symbols_per_step"])
    root = torch.nn.Module()
    for k, m in mods.items():
        root.add_module(k, m)
    root.load_state_dict(sd, strict=True)
    root.eval()
    return root, decoding
