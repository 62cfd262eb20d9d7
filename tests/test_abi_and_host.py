"""CPU: the C-ABI library loads and exports every symbol include/t2v.h declares (no compute calls), the
product refuses to run without CUDA, token indexing / collate are bit-exact restatements, reflection works on
the reference's dotted paths, losses match the oracle's restatement."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported_and_bound():
    from txt2vid_b200 import _lib
    lib = _lib.lib()
    with open(os.path.join(ROOT, "include", "t2v.h")) as f:
        declared = set(re.findall(r"\b(t2v_[a-z0-9_]+)\s*\(", f.read()))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SIGNATURES), sorted(declared ^ set(_lib.SIGNATURES))
    assert lib.t2v_version() >= 100


def test_no_cpu_fallback():
    from txt2vid_b200 import kernels as K
    from txt2vid_b200._lib import T2VError
    with pytest.raises(T2VError):
        K.relu_fwd(torch.zeros(16, dtype=torch.bfloat16))
    with pytest.raises(T2VError):
        K.conv_fprop(torch.zeros(1, 1, 1, 1, 16, dtype=torch.bfloat16), torch.zeros(16, 1, 16, dtype=torch.bfloat16),
                     k=(1, 1, 1))


def test_channel_reductions_reject_channel_counts_not_multiple_of_8():
    """the column reductions read 8 channels per load: C % 8 != 0 is refused before any CUDA call"""
    from txt2vid_b200 import _lib
    lib = _lib.lib()
    ERR_ARG = -1                                      # T2V_ERR_ARG of include/t2v.h
    for sfx in ("", "_f32"):
        assert getattr(lib, "t2v_sum_rows" + sfx)(None, None, 5, 12, None) == ERR_ARG
        assert getattr(lib, "t2v_sum_rows_acc" + sfx)(None, None, 5, 12, None) == ERR_ARG
        assert getattr(lib, "t2v_sum_spatial" + sfx)(None, None, 2, 3, 12, None) == ERR_ARG
        assert getattr(lib, "t2v_bn_stats" + sfx)(None, None, 5, 12, None) == ERR_ARG
        assert getattr(lib, "t2v_bn_bwd" + sfx)(None, None, None, None, None, None, 1, 1, 5, 12, 0, 1,
                                               None) == ERR_ARG


def test_environment_reads_are_diagnostics_and_launcher_variables_only():
    """The product reads no environment variable that selects a code path or a tuning value: what runs depends on
    the inputs and the code only.  Allowed are the diagnostics T2V_PROFILE_DUMP / T2V_DEBUG_LAUNCH (they print,
    select nothing) and the launcher's rank variables."""
    import glob
    pkg = os.path.join(ROOT, "txt2vid_b200")
    files = glob.glob(os.path.join(pkg, "**", "*.py"), recursive=True)
    files += [p for p in glob.glob(os.path.join(pkg, "csrc", "*")) if p.endswith((".cu", ".cuh", ".inc", ".h"))]
    files += glob.glob(os.path.join(ROOT, "include", "*.h"))
    read = re.compile(r"""\b(?:environ\.get|getenv|env_int)\s*\(\s*["']([^"']+)["']|\benviron\s*\[\s*["']([^"']+)["']""")
    names = set()
    for path in files:
        with open(path) as f:
            names.update(a or b for a, b in read.findall(f.read()))
    assert names == {"T2V_PROFILE_DUMP", "T2V_DEBUG_LAUNCH", "WORLD_SIZE", "RANK", "LOCAL_RANK"}, sorted(names)


def test_vocab_and_collate_bit_exact():
    from txt2vid_b200.data import Vocab, build_vocab, collate_fn
    sents = ["digit 3 is left and right.", "Digit 7 is top and bottom", "a man is cooking."]
    v = build_vocab(sents)
    assert [v(w) for w in (Vocab.PAD, Vocab.START, Vocab.END, Vocab.UNKNOWN)] == [0, 1, 2, 3]
    assert list(v.tokenize("digit 3 is left.")) == ["<start>", "digit", "3", "is", "left", "<end>"]
    a = v.encode(sents[0])
    b = v.encode(sents[1])                       # no trailing '.', END appended
    assert a[0] == 1 and a[-1] == 2 and b[-1] == 2 and v("zebra") == 3
    assert v.to_words(a) == "<start> digit 3 is left and right<end>"
    vids = [torch.zeros(2), torch.ones(2), torch.full((2,), 2.0)]
    caps = [v.encode(s) for s in sents]
    x, tok, lens = collate_fn(list(zip(vids, caps)))
    assert lens == sorted(lens, reverse=True) and tok.shape == (3, max(lens)) and tok.dtype == torch.int64
    for i, L in enumerate(lens):
        assert (tok[i, L:] == 0).all() and tok[i, L - 1] == 2


def test_vocab_and_collate_match_the_reference_fixtures():
    """SURVEY 8(a) row T against the reference's OWN Vocab / build_vocab / collate_fn and the caption part of
    Dataset.__getitem__ (data/__init__.py:250-254,260-355): tests/golden/token_fixtures.json was recorded from the live
    reference by oracle/make_golden_tokens.py (nvidia.dali stubbed).  Bit-exact: vocabulary, token ids, padded int64
    batches, sort order (stable, longest first), lengths, to_words round trip."""
    from helpers import golden
    from txt2vid_b200.data import build_vocab, collate_fn
    fx = golden("token_fixtures.json")
    v = build_vocab(fx["vocab_sentences"])
    assert v.word2idx == fx["word2idx"] and len(v) == fx["len"]
    enc = []
    for rec in fx["encoded"]:
        t = v.encode(rec["sentence"])
        assert t.dtype == torch.int64 and t.tolist() == rec["tokens"], rec["sentence"]
        assert v.to_words(t) == rec["words"]
        enc.append(t)
    for b in fx["batches"]:
        data = [(torch.full((2,), float(i)), enc[i]) for i in b["picks"]]
        vids, tok, lens = collate_fn(data)
        assert [int(x[0]) for x in vids] == b["order"]
        assert tok.dtype == torch.int64 and tok.tolist() == b["targets"] and [int(l) for l in lens] == b["lengths"]


def test_reflection_on_reference_paths():
    import contextlib
    import io
    from txt2vid_b200.util import count_params, create_object
    with contextlib.redirect_stdout(io.StringIO()):
        d = create_object({"class": "txt2vid.models.tganv2.discrim.MultiScaleDiscrim", "args": {"num_channels": 3}},
                          cond_dim=0)
        loss = create_object("txt2vid.gan.losses.RSGANLoss")
    assert count_params(d) == 29039746          # SURVEY.md section 6 (probed on the reference)
    assert hasattr(d, "sub_discrims") and len(d.sub_discrims) == 4 and hasattr(loss, "discrim_loss")


def test_losses_match_oracle(monkeypatch):
    """RSGAN / Wasserstein run on the fused reduction kernel (ops.rel_loss): here with the kernel's executable spec"""
    import cpu_kernels
    import oracle.txt2vid_oracle as O
    from txt2vid_b200 import gan, ops
    monkeypatch.setattr(ops, "K", cpu_kernels)
    torch.manual_seed(0)
    f, r = torch.randn(8, 1), torch.randn(8, 1)
    pairs = [(gan.RSGANLoss(), O.RSGAN), (gan.WassersteinGanLoss(), O.Wasserstein), (gan.RaLSGANLoss(), O.RaLSGAN),
             (gan.VanillaGanLoss(), O.Vanilla)]
    for mine, ref in pairs:
        assert torch.allclose(mine.discrim_loss(fake=f, real=r), ref.discrim_loss(f, r), atol=1e-6)
        assert torch.allclose(mine.gen_loss(fake=f, real=r), ref.gen_loss(f, r), atol=1e-6)
    with pytest.raises(AttributeError):
        gan.RaSGANLoss().discrim_loss(fake=f, real=r)
