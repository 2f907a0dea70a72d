"""TEST INFRASTRUCTURE.  Generates tests/golden/*.pt by executing the reference's OWN module files
(via oracle/ref_stub.py) on seeded synthetic inputs.  Run in the build container only:

    python oracle/make_golden.py

The fixtures are small (tiny config: 2 layers, d=256, ffn=1024, 4 heads — BASELINE.json configs[0])
and are committed; the GPU box never sees /root/reference.
"""
import math
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_stub  # noqa: E402
import synth  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def audio_pretrain():
    """tests/golden/pretrain_audio_criterion.pt: the audio-text pretraining criterion through the reference's own model +
    criterion files (one_peace_pretrain.py:106-179 with the audio preserve_ids gather adapter/audio.py:184-189 and the
    'fixed'-position decoder canvas :172-181; audio_text_pretrain_loss.py:73-208)."""
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    crit_mod = ref_stub.ref_module("one_peace.criterions.audio_text_pretrain_loss")
    pm = ref_stub.build_reference_audio_pretrain(**synth.PRETRAIN_AUDIO_TINY)
    psd = synth.make_audio_pretrain_state_dict(**synth.PRETRAIN_AUDIO_TINY, seed=0)
    missing, unexpected = pm.load_state_dict(psd, strict=False)
    assert not unexpected and all(k.endswith(("rp_bucket", "position_idx", "version")) for k in missing), (missing, unexpected)
    sample = synth.pretrain_audio_sample(seed=0, vocab=synth.PRETRAIN_AUDIO_TINY["vocab"])
    crit = crit_mod.AudioTextPretrainLossCriterion(task=None, dcl_audio_alpha=1.0, dcl_al_text_alpha=0.5, dcl_al_audio_alpha=0.5,
                                                   dcl_logit_scale=2.5, label_smoothing=0.1)
    for q in pm.parameters():
        q.requires_grad_(True)
    pm.zero_grad(set_to_none=True)
    loss, _, log = crit(pm, sample)
    loss.backward()
    ni = sample["net_input"]
    kw = dict(src_audios=ni["src_audios"], audio_padding_masks=ni["audio_padding_masks"])
    with torch.no_grad():
        _, _, dec_a = pm(audio_preserve_ids=ni["audio_preserve_ids"], encoder_type="audio", **kw)
        dat, _, daa = pm(src_tokens=ni["src_tokens"], text_preserve_ids=ni["al_text_preserve_ids"],
                         audio_preserve_ids=ni["al_audio_preserve_ids"], encoder_type="al", **kw)
        al, af = pm(encoder_type="audio", **kw)
        ax, apad, abias = pm.encoder_wrapper.audio_adapter(ni["src_audios"], ni["audio_padding_masks"],
                                                           preserve_ids=ni["audio_preserve_ids"])
    torch.save({"config": synth.PRETRAIN_AUDIO_TINY, "weights_seed": 0, "sample_seed": 0,
                "log": {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in log.items()},
                "student_audio": dec_a, "student_al_text": dat, "student_al_audio": daa, "audio_logits": al,
                "audio_features": af[:, :8].clone(), "adapter_student_x": ax, "adapter_student_bias": abias[0][:, :, :8, :8].clone(),
                "grads": {n: synth.grad_summary(n, q.grad) for n, q in pm.named_parameters() if q.grad is not None}},
               os.path.join(OUT, "pretrain_audio_criterion.pt"))
    print("pretrain_audio_criterion.pt", os.path.getsize(os.path.join(OUT, "pretrain_audio_criterion.pt")))


def main():
    if sys.argv[1:] == ["audio_pretrain"]:
        return audio_pretrain()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    cfgd = dict(embed_dim=256, ffn=1024, layers=2, heads=4)
    model = ref_stub.build_reference_retrieval(embed_dim=256, ffn=1024, layers=2, heads=4, head_type="val", seed=0,
                                               vocab=50264)
    sd = synth.make_state_dict(**cfgd, seed=0)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    # only deterministic buffers may be absent from the synthetic state dict
    assert not unexpected, unexpected
    assert all(k.endswith(("rp_bucket", "position_idx", "version")) for k in missing), missing
    tok, img, aud, apm = synth.tiny_inputs(seed=0)
    with torch.no_grad():
        text = model(src_tokens=tok, encoder_type="text")
        image = model(src_images=img, encoder_type="image")
        audio = model(src_audios=aud, audio_padding_masks=apm, encoder_type="audio")
        tx, tpad, tbias = model.encoder_wrapper.text_adapter(tok)
        ix, ipad, ibias = model.encoder_wrapper.image_adapter(img)
        ax, apad, abias = model.encoder_wrapper.audio_adapter(aud, apm)
        # layer-0 output of the text branch (transformer_layer.py:165-228 through the reference module)
        fm = model.encoder_wrapper.fusion_model
        x0 = (tx * (1 - tpad.unsqueeze(-1).type_as(tx))).transpose(0, 1)
        bias_full = tbias[0].contiguous().clone()
        bias_full.masked_fill_(tpad[:, None, None, :], float("-inf"))
        l0 = fm.layers[0](x0, encoder_padding_mask=tpad, self_attn_bias=bias_full, encoder_type="text",
                          text_seq_len=tx.size(1), image_seq_len=0, audio_seq_len=0).transpose(0, 1)
    torch.save({
        "config": cfgd, "weights_seed": 0, "inputs_seed": 0,
        "outputs": dict(text=text, image=image, audio=audio),
        "adapter": dict(text_x=tx, text_pad=tpad, text_bias=tbias[0][0], image_x=ix[:1].clone(), image_bias=ibias[0][0, :, :40, :40].clone(),
                        audio_x=ax, audio_bias=abias[0][0]),
    }, os.path.join(OUT, "tiny_retrieval.pt"))
    # a file of its own keeps every golden file under 1 MB
    torch.save({"config": cfgd, "weights_seed": 0, "inputs_seed": 0, "text_layer0_out": l0},
               os.path.join(OUT, "tiny_text_layer0.pt"))

    # ---- gradients of the reference modules (torch autograd through the reference's own forward) ----
    # Summaries only (norm, seeded random projection, first 256 elements per parameter): they pin the oracle's
    # backward (tests/test_oracle_golden.py), which in turn checks the hand-written CUDA backward on the GPU.
    for p in model.parameters():
        p.requires_grad_(True)
    gt = torch.Generator().manual_seed(100)
    targets = dict(text=torch.randn(8, 256, generator=gt), image=torch.randn(2, 256, generator=gt))
    grads = {}
    for modality, kw in (("text", dict(src_tokens=tok[:8])), ("image", dict(src_images=img))):
        model.zero_grad(set_to_none=True)
        emb = model(encoder_type=modality, **kw)
        (emb * targets[modality]).sum().backward()
        grads[modality] = {n: synth.grad_summary(n, p.grad) for n, p in model.named_parameters() if p.grad is not None}
    torch.save({"config": cfgd, "weights_seed": 0, "inputs_seed": 0, "targets_seed": 100, "n_text": 8, "grads": grads},
               os.path.join(OUT, "tiny_train_grads.pt"))
    model.zero_grad(set_to_none=True)

    # ---- contrastive head (criterion file executed as-is; single process: .data path) ----
    crit_mod = ref_stub.ref_module("one_peace.criterions.image_text_retrieval_loss")
    cases = []
    for (b, d, eps, seed) in [(16, 64, 0.0, 10), (48, 256, 0.1, 11), (128, 1536, 0.0, 12)]:
        img_e, txt_e = synth.contrastive_pair(b, d, seed)
        img_e.requires_grad_(True); txt_e.requires_grad_(True)
        ls = torch.tensor(math.log(1 / 0.07), requires_grad=True)
        crit = crit_mod.ImageTextRetrievalCriterion(task=None, label_smoothing=eps)
        scale = ls.exp()
        loss, i2t, t2i = crit.compute_itc_loss(img_e, txt_e, img_e.data, txt_e.data, scale)
        loss.backward()
        cases.append(dict(b=b, d=d, eps=eps, seed=seed, logit_scale=ls.detach().clone(), loss=loss.detach(),
                          i2t_ncorrect=i2t, t2i_ncorrect=t2i, grad_image=img_e.grad[:8].clone(),
                          grad_text=txt_e.grad[:8].clone(), grad_image_norm=img_e.grad.norm(), grad_text_norm=txt_e.grad.norm(),
                          grad_logit_scale=ls.grad.clone()))
    torch.save(cases, os.path.join(OUT, "itc_loss.pt"))

    # ---- concatenated encoders ('vl' / 'al', ModelWrapper.forward one_peace_base.py:68-129) and the DCL loss ----
    with torch.no_grad():
        vt, vi, _ = model.encoder_wrapper(src_tokens=tok[:2], src_images=img, encoder_type="vl")
        at, _, aa = model.encoder_wrapper(src_tokens=tok[2:4], src_audios=aud, audio_padding_masks=apm, encoder_type="al")
    pre_mod = ref_stub.ref_module("one_peace.criterions.image_text_pretrain_loss")
    crit = object.__new__(pre_mod.ImageTextPretrainLossCriterion)          # only the two scalars below are read (:187-208)
    crit.dcl_logit_scale, crit.label_smoothing = 2.5, 0.1
    gd = torch.Generator().manual_seed(31)
    stu = torch.randn(3, 9, 64, generator=gd, requires_grad=True)
    tea = stu.detach() + 0.7 * torch.randn(3, 9, 64, generator=gd)
    msk = torch.rand(3, 9, generator=gd) < 0.4
    msk[:, 0] = False
    padm = torch.zeros(3, 8, dtype=torch.bool)
    padm[1, 6:] = True
    msk[1, 7:] = False
    dcl_a = crit.compute_dcl_loss(stu, tea, msk)
    dcl_b = crit.compute_dcl_loss(stu, tea, msk, padm)
    dcl_b.backward()
    torch.save({"vl_text": vt, "vl_image": vi, "al_text": at, "al_audio": aa, "dcl": dict(seed=31, no_pad=dcl_a.detach(),
                with_pad=dcl_b.detach(), grad_norm=stu.grad.norm(), grad_head=stu.grad[0, 1:3].clone())},
               os.path.join(OUT, "pretrain_path.pt"))

    # ---- the full image-text pretraining criterion through the reference's own model + criterion files ----
    # (one_peace_pretrain.py:106-179 incl. preserve_ids gathers, decoder canvas, mask heads; image_text_pretrain_loss.py:76-208)
    pm = ref_stub.build_reference_pretrain(**synth.PRETRAIN_TINY)
    psd = synth.make_pretrain_state_dict(**synth.PRETRAIN_TINY, seed=0)
    missing, unexpected = pm.load_state_dict(psd, strict=False)
    assert not unexpected and all(k.endswith(("rp_bucket", "position_idx", "version")) for k in missing), (missing, unexpected)
    sample = synth.pretrain_sample(seed=0, res=synth.PRETRAIN_TINY["res"], vocab=synth.PRETRAIN_TINY["vocab"])
    pcrit = pre_mod.ImageTextPretrainLossCriterion(task=None, dcl_text_alpha=0.5, dcl_image_alpha=1.0, dcl_vl_text_alpha=0.5,
                                                   dcl_vl_image_alpha=0.5, dcl_logit_scale=2.5, label_smoothing=0.1)
    for q in pm.parameters():
        q.requires_grad_(True)
    pm.zero_grad(set_to_none=True)
    ploss, _, plog = pcrit(pm, sample)
    ploss.backward()
    ni = sample["net_input"]
    with torch.no_grad():
        dec_t, _, _ = pm(src_tokens=ni["src_tokens"], text_preserve_ids=ni["text_preserve_ids"], encoder_type="text")
        dvt, dvi, _ = pm(src_tokens=ni["src_tokens"], text_preserve_ids=ni["vl_text_preserve_ids"], src_images=ni["src_images"],
                         image_preserve_ids=ni["vl_image_preserve_ids"], encoder_type="vl")
        tl, tf = pm(src_tokens=ni["src_tokens"], encoder_type="text")
    torch.save({"config": synth.PRETRAIN_TINY, "weights_seed": 0, "sample_seed": 0,
                "log": {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in plog.items()},
                "student_text": dec_t, "student_vl_text": dvt, "student_vl_image": dvi, "text_logits": tl, "text_features": tf,
                "grads": {n: synth.grad_summary(n, q.grad) for n, q in pm.named_parameters() if q.grad is not None}},
               os.path.join(OUT, "pretrain_criterion.pt"))

    # ---- retrieval evaluation (metrics/recall.py executed as-is, single process) ----
    rec_mod = ref_stub.ref_module("one_peace.metrics.recall")
    rcases = []
    for (n_img, cap, dd, seed, noise) in [(40, 5, 64, 21, 0.8), (64, 3, 256, 22, 1.5)]:
        img_e, txt_e, img_ids, txt_ids = synth.retrieval_set(n_img, cap, dd, seed, noise)
        rec = rec_mod.Recall()
        rec.initialize(txt_ids, txt_e)
        for lo in range(0, n_img, 16):                  # batches, as the eval loop feeds them (image_text_retrieval.py:62-111)
            rec.compute(img_ids[lo:lo + 16], img_e[lo:lo + 16])
        log = rec.merge_results(output_predict=True)
        rcases.append(dict(n_img=n_img, cap=cap, d=dd, seed=seed, noise=noise, log=log))
    torch.save(rcases, os.path.join(OUT, "recall.pt"))

    # ---- python Adam (optim/adam.py executed as-is) ----
    # adam.py imports omegaconf (absent) and its apex-probing siblings at module scope: provide shells.
    # adam_fused.py / distributed_fused_adam.py / base_optimizer.py themselves import fine under the stub
    # (their apex imports are wrapped in try/except) except for base_optimizer's FairseqOptimizer base.
    import types
    om = types.ModuleType("omegaconf"); om.II = lambda x: None; om.OmegaConf = object
    sys.modules.setdefault("omegaconf", om)
    ref_adam = ref_stub.ref_module("one_peace.optim.adam")
    Adam = ref_adam.Adam
    g = torch.Generator().manual_seed(3)
    p0 = torch.randn(1000, generator=g)
    grads = [torch.randn(1000, generator=g) * (0.1 + i) for i in range(3)]
    out = {}
    for tag, dt in [("fp32", torch.float32), ("bf16", torch.bfloat16)]:
        p = torch.nn.Parameter(p0.clone().to(dt))
        opt = Adam([p], lr=1e-2, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.05)
        traj = []
        for gi in grads:
            p.grad = gi.clone().to(dt)
            opt.step()
            traj.append(p.detach().clone())
        st = opt.state[p]
        out[tag] = dict(p0=p0.clone().to(dt), grads=[gi.to(dt) for gi in grads], traj=traj, exp_avg=st["exp_avg"].clone(),
                        exp_avg_sq=st["exp_avg_sq"].clone(), lr=1e-2, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.05)
    torch.save(out, os.path.join(OUT, "adam.pt"))
    audio_pretrain()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
