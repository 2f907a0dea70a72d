"""Pins oracle/restated.py (the CPU oracle) against tests/golden/*.pt, which were produced by executing the
reference's own module files (oracle/make_golden.py).  CPU only."""
import math
import os

import pytest
import torch

import restated as R
import synth


@pytest.fixture(scope="module")
def tiny(golden_dir):
    fx = torch.load(os.path.join(golden_dir, "tiny_retrieval.pt"), weights_only=False)
    c = fx["config"]
    sd = synth.make_state_dict(**c, seed=fx["weights_seed"])
    cfg = R.OracleConfig(embed_dim=c["embed_dim"], ffn_embed_dim=c["ffn"], layers=c["layers"], attention_heads=c["heads"])
    tok, img, aud, apm = synth.tiny_inputs(seed=fx["inputs_seed"])
    return fx, sd, cfg, (tok, img, aud, apm)


def test_bucket_tables_match_reference_shapes():
    b = R.make_token_bucket_position(256)
    assert b.shape == (1024, 1024) and int(b.max()) == 2 * 256 + 1 and int(b[0, 0]) == 513
    i = R.make_image_bucket_position(14)
    assert i.shape == (197, 197) and int(i.max()) == 27 * 27 + 2


def test_text_adapter(tiny):
    fx, sd, cfg, (tok, _, _, _) = tiny
    x, pad, bias = R.text_adapter(sd, cfg, tok)
    assert torch.equal(pad, fx["adapter"]["text_pad"])
    torch.testing.assert_close(x, fx["adapter"]["text_x"], atol=1e-6, rtol=0)
    torch.testing.assert_close(bias, fx["adapter"]["text_bias"], atol=0, rtol=0)


def test_image_adapter(tiny):
    fx, sd, cfg, (_, img, _, _) = tiny
    x, pad, bias = R.image_adapter(sd, cfg, img)
    assert not pad.any()
    torch.testing.assert_close(x[:1], fx["adapter"]["image_x"], atol=2e-5, rtol=0)
    torch.testing.assert_close(bias[:, :40, :40], fx["adapter"]["image_bias"], atol=0, rtol=0)


def test_audio_adapter(tiny):
    fx, sd, cfg, (_, _, aud, apm) = tiny
    x, pad, bias = R.audio_adapter(sd, cfg, aud, apm)
    assert x.shape[1] == R.audio_frames(aud.shape[1], cfg.feature_encoder_spec) + 1
    torch.testing.assert_close(x, fx["adapter"]["audio_x"], atol=5e-5, rtol=1e-5)
    torch.testing.assert_close(bias, fx["adapter"]["audio_bias"], atol=0, rtol=0)


def test_text_layer0(tiny, golden_dir):
    fx, sd, cfg, (tok, _, _, _) = tiny
    l0 = torch.load(os.path.join(golden_dir, "tiny_text_layer0.pt"), weights_only=False)
    assert (l0["config"], l0["weights_seed"], l0["inputs_seed"]) == (fx["config"], fx["weights_seed"], fx["inputs_seed"])
    x, pad, bias = R.text_adapter(sd, cfg, tok)
    x = x * (1 - pad.unsqueeze(-1).type_as(x))
    y = R.encoder_layer(sd, cfg, x, bias, pad, "text", "encoder_wrapper.fusion_model.layers.0.")
    torch.testing.assert_close(y, l0["text_layer0_out"], atol=2e-5, rtol=1e-5)


@pytest.mark.parametrize("modality", ["text", "image", "audio"])
def test_extract_features(tiny, modality):
    fx, sd, cfg, (tok, img, aud, apm) = tiny
    out = R.extract_features(sd, cfg, modality, src_tokens=tok, src_images=img, src_audios=aud, audio_padding_masks=apm)
    want = fx["outputs"][modality]
    torch.testing.assert_close(out, want, atol=1e-5, rtol=0)
    torch.testing.assert_close(out.norm(dim=1), torch.ones(out.shape[0]), atol=1e-5, rtol=0)


@pytest.mark.parametrize("modality", ["text", "image"])
def test_backward_vs_reference_autograd(golden_dir, modality):
    """torch autograd through the restatement == torch autograd through the reference's own modules
    (tests/golden/tiny_train_grads.pt, written by oracle/make_golden.py): pins the oracle the CUDA backward is checked
    against."""
    fx = torch.load(os.path.join(golden_dir, "tiny_train_grads.pt"), weights_only=False)
    sd = synth.make_state_dict(**fx["config"], seed=fx["weights_seed"])
    tok, img, _, _ = synth.tiny_inputs(seed=fx["inputs_seed"])
    gt = torch.Generator().manual_seed(fx["targets_seed"])
    targets = dict(text=torch.randn(8, 256, generator=gt), image=torch.randn(2, 256, generator=gt))
    cfg = R.OracleConfig(embed_dim=256, ffn_embed_dim=1024, layers=2, attention_heads=4)
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    kw = dict(src_tokens=tok[:fx["n_text"]]) if modality == "text" else dict(src_images=img)
    (R.extract_features(sdg, cfg, modality, **kw) * targets[modality]).sum().backward()
    want = fx["grads"][modality]
    n = 0
    for name, ref in want.items():
        if ref["norm"] == 0:
            continue
        got = synth.grad_summary(name, sdg[name].grad)
        assert got["shape"] == ref["shape"], name
        assert abs(got["norm"] - ref["norm"]) <= 2e-4 * ref["norm"] + 1e-9, (name, got["norm"], ref["norm"])
        assert abs(got["proj"] - ref["proj"]) <= 2e-4 * ref["norm"] + 1e-9, (name, got["proj"], ref["proj"])
        torch.testing.assert_close(got["head"], ref["head"], rtol=2e-3, atol=2e-5 * ref["norm"] + 1e-9)
        n += 1
    assert n >= 45, n          # 2 layers x 21 + adapter + head parameters on the modality's path


def test_concatenated_encoders_vs_reference(tiny, golden_dir):
    """'vl' / 'al' sequences (text + image / text + audio through shared attention, per-modality FFN and final norm):
    oracle encoder_multi vs the reference's ModelWrapper.forward (tests/golden/pretrain_path.pt)."""
    fx, sd, cfg, (tok, img, aud, apm) = tiny
    ref = torch.load(os.path.join(golden_dir, "pretrain_path.pt"), weights_only=False)
    with torch.no_grad():
        tx, tp, tb = R.text_adapter(sd, cfg, tok[:2])
        ix, ip, ib = R.image_adapter(sd, cfg, img)
        vt, vi = R.encoder_multi(sd, cfg, [(tx, tp, tb, "text"), (ix, ip, ib, "image")])
        tx, tp, tb = R.text_adapter(sd, cfg, tok[2:4])
        ax, ap, ab = R.audio_adapter(sd, cfg, aud, apm)
        at, aa = R.encoder_multi(sd, cfg, [(tx, tp, tb, "text"), (ax, ap, ab, "audio")])
    for got, key in ((vt, "vl_text"), (vi, "vl_image"), (at, "al_text"), (aa, "al_audio")):
        torch.testing.assert_close(got, ref[key], atol=3e-5, rtol=1e-4)


def test_dcl_loss_vs_reference(golden_dir):
    ref = torch.load(os.path.join(golden_dir, "pretrain_path.pt"), weights_only=False)["dcl"]
    gd = torch.Generator().manual_seed(ref["seed"])
    stu = torch.randn(3, 9, 64, generator=gd, requires_grad=True)
    tea = stu.detach() + 0.7 * torch.randn(3, 9, 64, generator=gd)
    msk = torch.rand(3, 9, generator=gd) < 0.4
    msk[:, 0] = False
    padm = torch.zeros(3, 8, dtype=torch.bool)
    padm[1, 6:] = True
    msk[1, 7:] = False
    torch.testing.assert_close(R.dcl_loss(stu, tea, msk), ref["no_pad"], atol=1e-6, rtol=1e-6)
    loss = R.dcl_loss(stu, tea, msk, padm)
    torch.testing.assert_close(loss, ref["with_pad"], atol=1e-6, rtol=1e-6)
    loss.backward()
    torch.testing.assert_close(stu.grad.norm(), ref["grad_norm"], atol=1e-6, rtol=1e-5)
    torch.testing.assert_close(stu.grad[0, 1:3], ref["grad_head"], atol=1e-6, rtol=1e-5)


def test_recall_eval_vs_reference(golden_dir):
    """oracle recall_eval == the reference's Recall metric executed on the same synthetic retrieval sets."""
    for c in torch.load(os.path.join(golden_dir, "recall.pt"), weights_only=False):
        img, txt, img_ids, txt_ids = synth.retrieval_set(c["n_img"], c["cap"], c["d"], c["seed"], c["noise"])
        got = R.recall_eval(img_ids, img, txt_ids, txt)
        for k in ("txt_r1", "txt_r5", "txt_r10", "img_r1", "img_r5", "img_r10", "r_mean"):
            assert abs(got[k] - c["log"][k]) < 1e-9, (k, got[k], c["log"][k])
        assert 5.0 < c["log"]["txt_r1"] < 99.0                     # the synthetic set is neither trivial nor hopeless
        for row, iid in enumerate(img_ids.tolist()):
            assert got["predict_txt"][row].tolist() == c["log"]["predict_txt"][iid]


def test_itc_loss_and_grads(golden_dir):
    cases = torch.load(os.path.join(golden_dir, "itc_loss.pt"), weights_only=False)
    for c in cases:
        a, t = synth.contrastive_pair(c["b"], c["d"], c["seed"])
        a.requires_grad_(True); t.requires_grad_(True)
        ls = c["logit_scale"].clone().requires_grad_(True)
        loss, i2t, t2i = R.itc_loss(a, t, a.detach(), t.detach(), R.logit_scale_exp(ls), 0, c["eps"])
        loss.backward()
        torch.testing.assert_close(loss.detach(), c["loss"], atol=1e-6, rtol=1e-6)
        assert float(i2t) == float(c["i2t_ncorrect"]) and float(t2i) == float(c["t2i_ncorrect"])
        torch.testing.assert_close(a.grad[:8], c["grad_image"], atol=1e-7, rtol=1e-5)
        torch.testing.assert_close(t.grad[:8], c["grad_text"], atol=1e-7, rtol=1e-5)
        torch.testing.assert_close(a.grad.norm(), c["grad_image_norm"], atol=0, rtol=1e-5)
        torch.testing.assert_close(ls.grad, c["grad_logit_scale"], atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("tag", ["fp32", "bf16"])
def test_adam(golden_dir, tag):
    fx = torch.load(os.path.join(golden_dir, "adam.pt"), weights_only=False)[tag]
    p = fx["p0"].clone()
    m = torch.zeros(p.shape); v = torch.zeros(p.shape)
    for step, (g, want) in enumerate(zip(fx["grads"], fx["traj"]), start=1):
        p32 = p.float()
        R.adam_step(p32, g.float(), m, v, step, fx["lr"], fx["betas"][0], fx["betas"][1], fx["eps"], fx["weight_decay"])
        p = p32.to(p.dtype)          # optim/adam.py:250-251: copy back (round to bf16 when params are bf16)
        assert torch.equal(p, want)
    torch.testing.assert_close(m, fx["exp_avg"], atol=0, rtol=0)
    torch.testing.assert_close(v, fx["exp_avg_sq"], atol=0, rtol=0)


def test_clip_coefficient_matches_fairseq_known_answer():
    # fairseq/tests/test_fp16_optimizer.py:57-82 pins grad-norm 2.2361 for grads (w: 2*? ...) of a
    # Linear(1,1) step: ||[1, 2]|| = sqrt(5).  Same formula (norm, then clamp(max_norm / (norm + 1e-6), max=1)).
    norm, coef = R.clip_coefficient([torch.tensor([1.0]), torch.tensor([2.0])], max_norm=1.0)
    assert abs(norm - 2.2361) < 1e-4 and abs(coef - 1.0 / (math.sqrt(5) + 1e-6)) < 1e-7


def test_pretrain_model_and_criterion_match_the_reference(golden_dir):
    """oracle/restated.py's pretraining model (preserve_ids gathers, decoder canvas, mask heads) and the full
    image_text_pretrain_loss vs the reference's own one_peace_pretrain.py + image_text_pretrain_loss.py executed on the same
    synthetic weights and masked batch (oracle/make_golden.py): every loss term, the student features, every parameter gradient."""
    fx = torch.load(os.path.join(golden_dir, "pretrain_criterion.pt"), weights_only=False)
    T = synth.PRETRAIN_TINY
    assert fx["config"] == T
    sd = synth.make_pretrain_state_dict(**T, seed=fx["weights_seed"])
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    w = T["res"] // 16
    cfg = R.OracleConfig(embed_dim=T["embed_dim"], ffn_embed_dim=T["ffn"], layers=T["layers"], attention_heads=T["heads"],
                         image_bucket_size=w, image_rel_bucket_size=w)
    dcfg = R.OracleConfig(embed_dim=T["dec_dim"], ffn_embed_dim=T["dec_ffn"], layers=T["dec_layers"], attention_heads=T["dec_heads"],
                          image_bucket_size=w, image_rel_bucket_size=w)
    sample = synth.pretrain_sample(seed=fx["sample_seed"], res=T["res"], vocab=T["vocab"])
    ni = sample["net_input"]
    with torch.no_grad():
        st, _, _ = R.pretrain_forward(sd, cfg, dcfg, src_tokens=ni["src_tokens"], text_preserve_ids=ni["text_preserve_ids"],
                                      encoder_type="text")
        vt, vi, _ = R.pretrain_forward(sd, cfg, dcfg, src_tokens=ni["src_tokens"], text_preserve_ids=ni["vl_text_preserve_ids"],
                                       src_images=ni["src_images"], image_preserve_ids=ni["vl_image_preserve_ids"], encoder_type="vl")
        tl, tf = R.pretrain_forward(sd, cfg, dcfg, src_tokens=ni["src_tokens"], encoder_type="text")
    torch.testing.assert_close(st, fx["student_text"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(vt, fx["student_vl_text"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(vi, fx["student_vl_image"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(tl, fx["text_logits"], atol=1e-5, rtol=1e-4)
    torch.testing.assert_close(tf, fx["text_features"], atol=5e-5, rtol=1e-4)
    loss, terms = R.image_text_pretrain_loss(sdg, cfg, dcfg, ni, label_smoothing=0.1)
    for k in ("itc_loss", "dcl_text_loss", "dcl_image_loss", "dcl_vl_text_loss", "dcl_vl_image_loss"):
        torch.testing.assert_close(terms[k].detach(), fx["log"][k], atol=2e-5, rtol=2e-5)
    torch.testing.assert_close(loss.detach(), fx["log"]["loss"], atol=5e-5, rtol=2e-5)
    assert float(terms["i2t_ncorrect"]) == float(fx["log"]["i2t_ncorrect"]) and float(terms["t2i_ncorrect"]) == float(fx["log"]["t2i_ncorrect"])
    loss.backward()
    checked = 0
    for name, summ in fx["grads"].items():
        g = sdg[name].grad
        if summ["norm"] == 0.0:
            assert g is None or float(g.norm()) < 1e-7, name
            continue
        assert g is not None, name
        mine = synth.grad_summary(name, g)
        assert mine["shape"] == summ["shape"], name
        assert abs(mine["norm"] - summ["norm"]) <= 2e-4 * summ["norm"] + 1e-7, (name, mine["norm"], summ["norm"])
        torch.testing.assert_close(mine["head"], summ["head"], atol=2e-4 * summ["norm"] + 1e-7, rtol=2e-3)
        checked += 1
    assert checked > 100


def test_audio_pretrain_model_and_criterion_match_the_reference(golden_dir):
    """The audio twin: oracle/restated.py's audio student passes (frame features gathered by preserve_ids BEFORE the positional
    convolution, 'fixed'-position decoder canvas) and audio_text_pretrain_loss vs the reference's one_peace_pretrain.py +
    audio_text_pretrain_loss.py executed on the same synthetic weights and masked ragged batch (oracle/make_golden.py)."""
    fx = torch.load(os.path.join(golden_dir, "pretrain_audio_criterion.pt"), weights_only=False)
    T = synth.PRETRAIN_AUDIO_TINY
    assert fx["config"] == T
    sd = synth.make_audio_pretrain_state_dict(**T, seed=fx["weights_seed"])
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    cfg = R.OracleConfig(embed_dim=T["embed_dim"], ffn_embed_dim=T["ffn"], layers=T["layers"], attention_heads=T["heads"])
    dcfg = R.OracleConfig(embed_dim=T["dec_dim"], ffn_embed_dim=T["dec_ffn"], layers=T["dec_layers"], attention_heads=T["dec_heads"])
    ni = synth.pretrain_audio_sample(seed=fx["sample_seed"], vocab=T["vocab"])["net_input"]
    kw = dict(src_audios=ni["src_audios"], audio_padding_masks=ni["audio_padding_masks"])
    with torch.no_grad():
        ax, apad, abias = R.audio_adapter_general(sd, cfg, ni["src_audios"], ni["audio_padding_masks"], ni["audio_preserve_ids"])
        _, _, sa = R.pretrain_forward(sd, cfg, dcfg, audio_preserve_ids=ni["audio_preserve_ids"], encoder_type="audio", **kw)
        sat, _, saa = R.pretrain_forward(sd, cfg, dcfg, src_tokens=ni["src_tokens"], text_preserve_ids=ni["al_text_preserve_ids"],
                                         audio_preserve_ids=ni["al_audio_preserve_ids"], encoder_type="al", **kw)
        al, af = R.pretrain_forward(sd, cfg, dcfg, encoder_type="audio", **kw)
    torch.testing.assert_close(ax, fx["adapter_student_x"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(abias[:, :, :8, :8], fx["adapter_student_bias"], atol=0, rtol=0)
    assert torch.equal(apad, ni["audio_preserve_ids"].eq(-1))
    torch.testing.assert_close(sa, fx["student_audio"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(sat, fx["student_al_text"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(saa, fx["student_al_audio"], atol=5e-5, rtol=1e-4)
    torch.testing.assert_close(al, fx["audio_logits"], atol=1e-5, rtol=1e-4)
    torch.testing.assert_close(af[:, :8], fx["audio_features"], atol=5e-5, rtol=1e-4)
    loss, terms = R.audio_text_pretrain_loss(sdg, cfg, dcfg, ni, label_smoothing=0.1)
    for k in ("atc_loss", "dcl_audio_loss", "dcl_al_text_loss", "dcl_al_audio_loss"):
        torch.testing.assert_close(terms[k].detach(), fx["log"][k], atol=2e-5, rtol=2e-5)
    torch.testing.assert_close(loss.detach(), fx["log"]["loss"], atol=5e-5, rtol=2e-5)
    assert float(terms["a2t_ncorrect"]) == float(fx["log"]["a2t_ncorrect"]) and float(terms["t2a_ncorrect"]) == float(fx["log"]["t2a_ncorrect"])
    loss.backward()
    checked = 0
    for name, summ in fx["grads"].items():
        g = sdg[name].grad
        if summ["norm"] == 0.0:
            assert g is None or float(g.norm()) < 1e-7, name
            continue
        assert g is not None, name
        mine = synth.grad_summary(name, g)
        assert mine["shape"] == summ["shape"], name
        assert abs(mine["norm"] - summ["norm"]) <= 2e-4 * summ["norm"] + 1e-7, (name, mine["norm"], summ["norm"])
        torch.testing.assert_close(mine["head"], summ["head"], atol=2e-4 * summ["norm"] + 1e-7, rtol=2e-3)
        checked += 1
    assert checked > 100
