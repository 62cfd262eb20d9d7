"""CPU: host-side pieces added around the kernels -- checkpoint compatibility with the reference (SURVEY 8f3), the
position-pair identity behind the small-channel weight gradients, lagged loss logging, the prefetcher's CPU path."""
import os

import pytest
import torch
import torch.nn.functional as F

from helpers import build_product_models, golden


def test_checkpoint_roundtrip_through_cond_gan(tmp_path):
    """CondGan.save_dict / load_from_dict (gan/cond_gan.py:186-217): keys gen / cond / <discriminator name>, the
    discriminator's parameters under `single_discrim.module.*`; torch.save -> torch.load -> fresh modules, exact."""
    from txt2vid_b200.gan import CondGan
    txt, gen, dis = build_product_models(True, V=50, seed=3)
    gan = CondGan(gen=gen, discrims=[dis], cond_encoder=txt, discrim_names=["video"])
    path = str(tmp_path / "iter_1")
    torch.save(gan.save_dict(), path)
    loaded = torch.load(path)
    assert set(loaded) == {"gen", "cond", "video"}
    assert any(k.startswith("single_discrim.module.") for k in loaded["video"])
    txt2, gen2, dis2 = build_product_models(True, V=50, seed=4)
    gan2 = CondGan(gen=gen2, discrims=[dis2], cond_encoder=txt2, discrim_names=["video"])
    gan2.load_from_dict(loaded)
    for a, b in ((gen, gen2), (dis, dis2), (txt, txt2)):
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa) == list(sb)
        assert all(torch.equal(sa[k], sb[k]) for k in sa)


def test_state_dicts_interchange_with_the_reference_modules():
    """A reference checkpoint's tensors line up with the product modules (models/tganv2_cond/{gen,discrim}.py,
    models/txt/basic.py): every floating-point state_dict entry the reference's modules recorded in the golden fixture
    (oracle/make_golden.py), with the same name, in the same order, with the same element count; and a product
    checkpoint loads back strictly into fresh product modules."""
    fx = golden("tganv2_cond_B8.json")
    txt, gen, dis = build_product_models(True, V=fx["config"]["V"], seed=fx["config"]["seed"])
    txt2, gen2, dis2 = build_product_models(True, V=fx["config"]["V"], seed=fx["config"]["seed"] + 1)
    for part, prod, fresh in (("gen", gen, gen2), ("dis", dis, dis2), ("txt", txt, txt2)):
        ref = fx["init"][part]
        sp = prod.state_dict()
        mine = [(k, v) for k, v in sp.items() if v.dtype.is_floating_point]
        assert [k for k, _ in mine] == list(ref), part
        assert all(v.numel() == ref[k]["n"] for k, v in mine), part
        fresh.load_state_dict(sp, strict=True)
        sf = fresh.state_dict()
        assert list(sf) == list(sp)
        assert all(sf[k].shape == sp[k].shape and torch.equal(sf[k], sp[k]) for k in sp)


def test_position_pair_identity_of_small_channel_weight_gradients():
    """kernels.conv_wgrad runs 32-channel (1,3,3) weight gradients on PAIRS of adjacent w voxels (64-channel views)
    and folds dw2[(pw,co)][a_h, s][(qw,ci)] into the real taps: shift a_w - 1 = 2 s + qw - pw (t2v_wgrad_fold_pairs).
    Here the same algebra in plain torch against the direct weight gradient."""
    g = torch.Generator().manual_seed(0)
    N, H, W, Ci, Co = 3, 6, 8, 4, 5
    x = torch.randn(N, H, W, Ci, generator=g, dtype=torch.float64)
    dy = torch.randn(N, H, W, Co, generator=g, dtype=torch.float64)
    direct = torch.nn.grad.conv2d_weight(x.permute(0, 3, 1, 2), (Co, Ci, 3, 3), dy.permute(0, 3, 1, 2), padding=1)
    x2, dy2 = x.reshape(N, H, W // 2, 2 * Ci), dy.reshape(N, H, W // 2, 2 * Co)
    dw2 = torch.nn.grad.conv2d_weight(x2.permute(0, 3, 1, 2), (2 * Co, 2 * Ci, 3, 3), dy2.permute(0, 3, 1, 2), padding=1)
    folded = torch.zeros_like(direct)
    for a_w in range(3):
        for s in (-1, 0, 1):
            for pw in (0, 1):
                for qw in (0, 1):
                    if 2 * s + qw - pw == a_w - 1:
                        folded[:, :, :, a_w] += dw2[pw * Co:(pw + 1) * Co, qw * Ci:(qw + 1) * Ci, :, s + 1]
    assert torch.allclose(folded, direct, rtol=1e-12, atol=1e-12)


def test_lagged_losses_cpu_path_is_immediate():
    from txt2vid_b200.trainer import LaggedLosses
    seen = []
    ll = LaggedLosses(lambda d, g: seen.append((d, g)), lag=2, device="cpu")
    ll.push(torch.tensor(1.5), torch.tensor(2.5))
    assert seen == [(1.5, 2.5)]
    ll.drain()
    assert seen == [(1.5, 2.5)]


def test_prefetcher_cpu_path_and_deferred_preload():
    """data_prefetcher on a CPU device is a plain iterator; next(preload=False) + preload() deliver the same batches."""
    from txt2vid_b200.data import data_prefetcher
    batches = [(torch.full((2, 3), float(i)), torch.full((2, 4), i, dtype=torch.long), [4, 4]) for i in range(5)]
    for deferred in (False, True):
        pf = data_prefetcher(iter(batches), device="cpu")
        got = []
        x, y = pf.next(preload=not deferred)
        while x is not None:
            got.append((float(x[0, 0]), int(y[0][0, 0]), y[1]))
            if deferred:
                pf.preload()
            x, y = pf.next(preload=not deferred)
        assert got == [(float(i), i, [4, 4]) for i in range(5)]


def test_caption_pretraining_step_matches_the_reference(monkeypatch):
    """SURVEY 8(f4): one step of train/txt.py:166-181 (encode -> teacher-forced / greedy decode -> cross entropy) on
    the weights and sentences of the fixture recorded from the reference (oracle/make_golden_caption_pretrain.py):
    same loss, the same decoded symbols in both modes, every parameter's gradient within 1e-4 (norm and probe).  The
    product's embedding / LSTM recurrence / GEMM kernels are replaced by their executable spec (tests/cpu_kernels.py,
    fp32 storage): this checks the host logic and the autograd formulas of text.py against the reference."""
    import cpu_kernels
    from test_round2_gpu import _golden_caption, _probe_index
    from txt2vid_b200 import ops
    from txt2vid_b200.text import Seq2Seq
    from txt2vid_b200.train_txt import pretrain_step
    monkeypatch.setattr(ops, "K", cpu_kernels)
    cpu_kernels.set_store_dtype(torch.float32)
    ops.PACKS.clear()
    try:
        fx = _golden_caption()
        torch.manual_seed(fx["seed"])
        prod = Seq2Seq(vocab_size=fx["V"])
        for n, p in prod.state_dict().items():
            s, a = fx["weights"][n]
            assert abs(float(p.double().sum()) - s) <= 1e-9 * max(1.0, a), n
        sent = torch.tensor(fx["sent"], dtype=torch.long)
        for mode, tf in (("teacher_force", True), ("greedy", False)):
            want = fx["modes"][mode]
            loss_p, sym_p = pretrain_step(prod, sent, fx["lengths"], None, teacher_force=tf)
            assert abs(float(loss_p) - want["loss"]) <= 2e-6 * abs(want["loss"]), (mode, float(loss_p), want["loss"])
            assert sym_p.tolist() == want["symbols"], mode
            for n, p in prod.named_parameters():
                g, w = p.grad.detach().reshape(-1), want["grads"][n]
                assert abs(float(g.double().norm()) - w["norm"]) <= 1e-4 * (w["norm"] + 1e-12), (mode, n)
                probe = torch.tensor(w["probe"])
                assert float((g[_probe_index(g.numel())] - probe).norm()) <= 1e-4 * (float(probe.norm()) + 1e-12), \
                    (mode, n)
    finally:
        cpu_kernels.set_store_dtype(torch.bfloat16)
        ops.PACKS.clear()


def test_caption_pretraining_golden_fixture_through_the_executable_spec(monkeypatch):
    """The committed fixture of oracle/make_golden_caption_pretrain.py (recorded from the live reference) against the
    product's host logic + autograd formulas on the CPU spec kernels (fp32): the same check the GPU test
    test_round2_gpu.py::test_caption_pretraining_step_vs_reference_golden runs through the real kernels."""
    import cpu_kernels
    from txt2vid_b200 import ops
    monkeypatch.setattr(ops, "K", cpu_kernels)
    cpu_kernels.set_store_dtype(torch.float32)
    ops.PACKS.clear()
    try:
        from test_round2_gpu import run_caption_pretrain_against_golden
        rep = run_caption_pretrain_against_golden("cpu", 1e-5, 1e-4, 1e-3)
        assert rep["teacher_force"]["loss"] < 1e-5
    finally:
        cpu_kernels.set_store_dtype(torch.bfloat16)
        ops.PACKS.clear()


@pytest.fixture()
def emulated_fp32(monkeypatch):
    import cpu_kernels
    from txt2vid_b200 import ops, optim, trainer
    for mod in (ops, optim, trainer):
        monkeypatch.setattr(mod, "K", cpu_kernels)
    monkeypatch.setattr(ops, "BF16", torch.float32)
    cpu_kernels.set_store_dtype(torch.float32)
    ops.PACKS.clear()
    yield
    cpu_kernels.set_store_dtype(torch.bfloat16)
    ops.PACKS.clear()


def test_trainer_test_writes_the_reference_sample_files(tmp_path, emulated_fp32):
    """SURVEY 8(f2): trainer.test() (gan/trainer.py:44-90) -- eval-mode generator, ONE full-resolution clip per
    sample, the reference's file names: real_<i>.png, sentences_<i>_<j>.txt (vocab.to_words of the token rows),
    <h>x<w>_<i>_<j>.jpg.  Host logic on the kernels' executable spec."""
    from types import SimpleNamespace
    from txt2vid_b200.data import build_vocab, collate_fn
    from txt2vid_b200.gan import CondGan
    from txt2vid_b200.trainer import test as run_test
    sents = ["digit 3 is left and right.", "digit 7 is top and bottom."]
    vocab = build_vocab(sents)
    txt, gen, dis = build_product_models(True, V=len(vocab), seed=5)
    gan = CondGan(gen=gen, discrims=[dis], cond_encoder=txt, discrim_names=["video"])
    g = torch.Generator().manual_seed(0)
    vids = [torch.rand(16, 3, 64, 64, generator=g) * 2 - 1 for _ in sents]          # loader order (T, C, H, W)
    batch = collate_fn([(v, vocab.encode(s)) for v, s in zip(vids, sents)])
    params = SimpleNamespace(out_samples=str(tmp_path / "samples"), img_model=False)
    run_test(gan=gan, num_samples=2, dataset=[batch], device=torch.device("cpu"), params=params, vocab=vocab)
    assert not gan.gen.training
    names = sorted(os.listdir(params.out_samples))
    assert names == ["64x64_0_0.jpg", "64x64_1_0.jpg", "real_0.png", "real_1.png", "sentences_0_0.txt",
                     "sentences_1_0.txt"], names
    with open(os.path.join(params.out_samples, "sentences_0_0.txt")) as f:
        lines = f.read().splitlines()
    assert lines == ["<start> digit 3 is left and right<end>", "<start> digit 7 is top and bottom<end>"]
    from PIL import Image
    im = Image.open(os.path.join(params.out_samples, "64x64_0_0.jpg"))
    assert im.size == (16 * 64 + 17 * 2, 2 * 64 + 3 * 2)                             # nrow = 16 frames, 2 clips, padding 2

