"""Golden fixtures from the REAL reference MODULES (not just leaf helpers), run in the build container:

    python oracle/gen_golden_modules.py            # writes tests/golden/ref_*.pt

oracle/ref_import.py mounts /root/reference/projects/HIPIE/hipie so that the unmodified reference files execute here
(their absent third-party packages are stubbed; the MSDeformAttn pybind op is bound to the reference's own
ms_deform_attn_core_pytorch).  Each fixture = seeded inputs + the reference module's state_dict + its outputs at a small
size; tests/test_oracle_modules.py loads the state_dict into the oracle's restatement of the same module and requires the
same outputs, which pins these rows of SURVEY.md §8a to the reference itself:

  ref_vit.pt          a2-a4   backbone/vit.py ViT.forward (PatchEmbed, abs-pos, windowed + global Block/Attention, FPN)
  ref_transformer.pt  a8-a13  deformable_transformer_dino.py DeformableTransformerVLDINO.forward (VLFuse, encoder layers with
                              MSDeformAttn.forward, two-stage proposals, bg queries, decoder layers, look-forward-twice refs)
  ref_heads.pt        a14-a15 deformable_detr.py VL_Align / Still_Classifier / MLP
  ref_maskdino.pt     a17-a19 maskdino_encoder.py MaskDINOEncoder.forward_features, maskdino_decoder.py MaskDINODecoder.forward
                              (+ dino_decoder.py TransformerDecoder, forward_prediction_heads with the mask-embed einsum)
  ref_condinst.pt     a16     ddetrs_dn.py dynamic_mask_with_coords / mask_heads_forward / parse_dynamic_params /
                              compute_locations / aligned_bilinear, MaskHeadSmallConv.forward
  ref_bert_chunk.pt   a7      bert_model.py BertEncoder.forward incl. the > 512-token chunk path (random-init HF BertModel)
  ref_postproc.pt     a20-a23 hipie_img.py convert_grounding_to_od_logits / semantic_inference / panoptic_inference,
                              ddetrs.py segmentation_postprocess
  ref_maskclip.pt     a22/f2  open_vocab/clip.py MaskCLIP (mask tokens, per-query attention masks, logit ensembling) and ClipAdapter._encode_text
                              on top of the restated open_clip 2.0.2 model (absent third-party dependency: hipie_oracle/clip.py), and
                              hipie_img.py HIPIE_IMG.get_clip_logits (MUL and ADD fusion, seen / unseen weights)
  ref_configs.json            projects/HIPIE/configs: the r50 / ViT-H training and ADE eval YAMLs with their _BASE_ and MaskDINO
                              config chains (the config surface, hipie_b200/config.py, has to load them unchanged)
  ref_msda_binding.pt a12     ops/functions/ms_deform_attn_func.py: MSDeformAttnFunction's call of the pybind op (argument order)
                              and ms_deform_attn_core_pytorch on the same inputs
"""
import copy
import os
import sys
import types

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, ".."))
import ref_import  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")


from hipie_oracle.synth import fill_by_name_  # noqa: E402


def randomize_(module, seed):
    """weights = a deterministic function of (parameter name, shape, seed): the fixtures carry inputs and outputs only and the
    test re-creates the same weights in the oracle's restatement through the same names (hipie_oracle.synth.fill_by_name_)"""
    return fill_by_name_(module, seed)


def small_cfg():
    from hipie_b200.config import add_hipie_config, get_cfg
    cfg = get_cfg()
    add_hipie_config(cfg)
    m = cfg.MODEL
    m.DECOUPLE_TGT, m.STILL_TGT_FOR_BOTH, m.VL_FUSION_USE_CHECKPOINT = True, True, False
    m.DDETRS.HIDDEN_DIM, m.DDETRS.VL_HIDDEN_DIM, m.DDETRS.ENC_LAYERS, m.DDETRS.DEC_LAYERS = 256, 64, 2, 2
    m.DDETRS.TWO_STAGE_NUM_BG_PROPOSALS, m.DDETRS.NUM_VL_LAYERS = 3, 1
    m.LANGUAGE_BACKBONE.LANG_DIM = 768      # the transformer's resizer hard-codes 768 (deformable_transformer_dino.py:99-103)
    return cfg


def gen_vit():
    vit = ref_import.ref("backbone.vit")
    torch.manual_seed(1)
    kw = dict(img_size=64, patch_size=16, embed_dim=32, depth=3, num_heads=2, use_rel_pos=True, window_size=14,
              window_block_indexes=(0, 2), pretrain_img_size=224, out_feature="last_feat")
    m = randomize_(vit.ViT(**kw), 2).eval()
    x = torch.randn(2, 3, 96, 80)
    with torch.no_grad():
        out = m(x)
    torch.save(dict(kw=dict(embed_dim=32, depth=3, num_heads=2, window_size=14, window_block_indexes=(0, 2), img_size=64, patch_size=16,
                            pretrain_img_size=224),
                    seed=2, keys=sorted(m.state_dict().keys()), x=x, out=out), os.path.join(OUT, "ref_vit.pt"))
    print("ref_vit.pt", {k: tuple(v.shape) for k, v in out.items()})


def _attach_heads(tr, dd, cfg, d, nd):
    """what DeformableDETR.__init__ does to the transformer (deformable_detr.py:262-292): per-layer VL_Align / MLP clones,
    Still_Classifier as the encoder-proposal scorer"""
    class_embed = dd.VL_Align(cfg)
    bbox_embed = dd.MLP(d, d, 4, 3)
    tr.decoder.class_embed = nn.ModuleList([copy.deepcopy(class_embed) for _ in range(nd + 1)])
    tr.decoder.bbox_embed = nn.ModuleList([copy.deepcopy(bbox_embed) for _ in range(nd + 1)])
    tr.decoder.class_embed[-1] = dd.Still_Classifier(d)


def gen_transformer():
    cfg = small_cfg()
    tmod = ref_import.ref("models.deformable_detr.deformable_transformer_dino")
    dd = ref_import.ref("models.deformable_detr.deformable_detr")
    torch.manual_seed(3)
    d, nd = 256, 2      # 256: the decoder's ref_point_head consumes 4 x 128 sine features (hard-coded)
    tr = tmod.DeformableTransformerVLDINO(d_model=d, nhead=8, num_encoder_layers=2, num_decoder_layers=nd, dim_feedforward=40, dropout=0.0,
                                          activation="relu", return_intermediate_dec=True, num_feature_levels=4, dec_n_points=4,
                                          enc_n_points=4, two_stage=True, two_stage_num_proposals=12, look_forward_twice=True,
                                          mixed_selection=True, use_checkpoint=False, cfg=cfg)
    _attach_heads(tr, dd, cfg, d, nd)
    randomize_(tr, 4).eval()
    g = torch.Generator().manual_seed(5)
    shapes = [(12, 10), (6, 5), (3, 3), (2, 2)]
    srcs = [torch.randn(2, d, h, w, generator=g) for h, w in shapes]
    masks = []
    for h, w in shapes:
        mk = torch.zeros(2, h, w, dtype=torch.bool)
        mk[1, h - max(1, h // 4):, :] = True          # image 1 is padded at the bottom and on the right
        mk[1, :, w - max(1, w // 5):] = True
        masks.append(mk)
    masks[3][1] = False
    masks[3][1, 1:, :] = True
    poses = [torch.randn(2, d, h, w, generator=g) for h, w in shapes]
    lang = {"hidden": torch.randn(2, 9, 768, generator=g), "masks": torch.ones(2, 9, dtype=torch.long)}
    lang["masks"][1, 6:] = 0
    lang_in = {k: v.clone() for k, v in lang.items()}
    with torch.no_grad():
        hs, memory, init_ref, inter_refs, enc_cls, enc_coord, lang_out = tr(
            srcs, masks, poses, query_embed=(None, None), mask_on=True, language_dict_features=lang, task="detection")
    torch.save(dict(seed=4, keys=sorted(tr.state_dict().keys()), srcs=srcs, masks=masks, poses=poses, lang=lang_in, hs=hs, memory=memory, init_ref=init_ref,
                    inter_refs=inter_refs, enc_cls=enc_cls, enc_coord=enc_coord, lang_hidden=lang_out["hidden"],
                    kw=dict(d_model=d, nhead=8, num_encoder_layers=2, num_decoder_layers=nd, dim_feedforward=40, two_stage_num_proposals=12,
                            num_bg=3, vl_hidden=64, lang_dim=768)),
               os.path.join(OUT, "ref_transformer.pt"))
    print("ref_transformer.pt hs", tuple(hs.shape), "memory", tuple(memory.shape))
    # heads
    torch.manual_seed(6)
    va = randomize_(dd.VL_Align(cfg), 7).eval()
    with torch.no_grad():
        va.log_scale.fill_(0.3)
    q = torch.randn(2, 5, d, generator=g)
    emb = torch.randn(2, 9, 768, generator=g)
    mlp = randomize_(dd.MLP(d, d, 4, 3), 8).eval()
    with torch.no_grad():
        torch.save(dict(va_seed=7, mlp_seed=8, q=q, emb=emb, va_out=va(q, emb), mlp_out=mlp(q)),
                   os.path.join(OUT, "ref_heads.pt"))
    print("ref_heads.pt")


def gen_maskdino():
    enc_mod = ref_import.ref("models.maskdino.pixel_decoder.maskdino_encoder")
    dec_mod = ref_import.ref("models.maskdino.transformer_decoder.maskdino_decoder")
    from detectron2.layers import ShapeSpec
    torch.manual_seed(9)
    c3, c4, c5, d = 24, 40, 40, 256       # 256: dino_decoder's ref_point_head consumes 4 x 128 sine features (hard-coded)
    enc = enc_mod.MaskDINOEncoder(
        {"res3": ShapeSpec(channels=c3, stride=8), "res4": ShapeSpec(channels=c4, stride=16), "res5": ShapeSpec(channels=c5, stride=32)},
        transformer_dropout=0.0, transformer_nheads=8, transformer_dim_feedforward=48, transformer_enc_layers=2, conv_dim=d, mask_dim=d,
        norm="GN", transformer_in_features=["res3", "res4", "res5"], common_stride=4, num_feature_levels=3, total_num_feature_levels=4,
        feature_order="low2high")
    randomize_(enc, 10).eval()
    g = torch.Generator().manual_seed(11)
    feats = {"res3": torch.randn(2, c3, 12, 16, generator=g), "res4": torch.randn(2, c4, 6, 8, generator=g),
             "res5": torch.randn(2, c5, 3, 4, generator=g)}
    with torch.no_grad():
        mask_features, out0, multi_scale = enc.forward_features(feats, None)
    dec = dec_mod.MaskDINODecoder(d, True, num_classes=d, hidden_dim=d, num_queries=7, nheads=8, dim_feedforward=48, dec_layers=3, mask_dim=d,
                                  enforce_input_project=False, two_stage=True, dn="seg", noise_scale=0.4, dn_num=100,
                                  initialize_box_type="no", initial_pred=True, learn_tgt=False, total_num_feature_levels=4, dropout=0.0)
    randomize_(dec, 12).eval()
    with torch.no_grad():
        out, _ = dec(multi_scale, mask_features, None)
    torch.save(dict(enc_seed=10, dec_seed=12, enc_keys=sorted(enc.state_dict().keys()), dec_keys=sorted(dec.state_dict().keys()),
                    in_channels=(c3, c4, c5), feats=feats, mask_features=mask_features, multi_scale=multi_scale,
                    pred_logits=out["pred_logits"], pred_masks=out["pred_masks"], pred_boxes=out["pred_boxes"],
                    interm_masks=out["interm_outputs"]["pred_masks"], interm_boxes=out["interm_outputs"]["pred_boxes"]),
               os.path.join(OUT, "ref_maskdino.pt"))
    print("ref_maskdino.pt", tuple(out["pred_masks"].shape), tuple(mask_features.shape))


def gen_condinst():
    dn = ref_import.ref("models.ddetrs_dn")
    torch.manual_seed(13)
    g = torch.Generator().manual_seed(14)
    head = randomize_(dn.MaskHeadSmallConv(256, None, 256), 15).eval()
    enc = [torch.randn(2, 256, 12, 16, generator=g), torch.randn(2, 256, 6, 8, generator=g), torch.randn(2, 256, 3, 4, generator=g)]
    with torch.no_grad():
        decod = head(enc, fpns=None)                           # (2, 8, 12, 16)
    fake = types.SimpleNamespace(no_rel_pos=False, dynamic_mask_channels=8, weight_nums=[80, 64, 8], bias_nums=[8, 8, 1], mask_out_stride=4,
                                 use_raft=False)
    fake.mask_heads_forward = lambda *a: dn.DDETRSegmUniDN.mask_heads_forward(fake, *a)
    nq = 5
    params = torch.randn(2, nq, 169, generator=g)
    ref_px = torch.rand(2, nq, 2, generator=g) * torch.tensor([128.0, 96.0])
    with torch.no_grad():
        logits = dn.DDETRSegmUniDN.dynamic_mask_with_coords(fake, decod, ref_px.reshape(1, 2 * nq, 2), params.reshape(1, 2 * nq, 169),
                                                            num_insts=[nq, nq], mask_feat_stride=8, rel_coord=True, up_masks=None)
    x = torch.randn(3, 1, 5, 7, generator=g)
    torch.save(dict(head_seed=15, head_keys=sorted(head.state_dict().keys()), enc=enc, decod=decod, params=params, ref_px=ref_px,
                    logits=logits.reshape(2, nq, logits.shape[-2], logits.shape[-1]), ab_in=x, ab_out=dn.aligned_bilinear(x, 2),
                    locations=dn.compute_locations(3, 4, device="cpu", stride=8)),
               os.path.join(OUT, "ref_condinst.pt"))
    print("ref_condinst.pt", tuple(logits.shape))


def gen_bert():
    """BertEncoder.forward with a 1300-token prompt (chunk path) and a 40-token prompt (plain path) on a random-init 2-layer HF
    BertModel: `from_pretrained` of the absent checkpoint directory is redirected to a seeded random model."""
    import transformers
    bm = ref_import.ref("models.deformable_detr.bert_model")
    conf = transformers.BertConfig(vocab_size=30522, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=96,
                                   max_position_embeddings=512, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    bm.BertConfig.from_pretrained = classmethod(lambda cls, *a, **k: conf)
    bm.BertModel.from_pretrained = classmethod(lambda cls, *a, config=None, add_pooling_layer=False, **k: cls(config, add_pooling_layer=add_pooling_layer))
    cfg = small_cfg()
    cfg.MODEL.LANGUAGE_BACKBONE.MAX_QUERY_LEN = 2048
    torch.manual_seed(16)
    enc = bm.BertEncoder(cfg)
    randomize_(enc, 17).eval()
    from hipie_oracle import synth
    ids, am, _, _ = synth.make_text(430, 2048, seed=18)
    assert int(am.sum()) > 1024
    ids = torch.cat([ids, ids.flip(0)[:, :1].expand(1, 2048) * 0 + ids], 0)           # batch of 2 (same prompt)
    am = torch.cat([am, am], 0)
    ids2, am2, _, _ = synth.make_text(12, 64, seed=19)
    with torch.no_grad():
        long = enc({"input_ids": ids, "attention_mask": am}, task="detection", sep=1012)
        short = enc({"input_ids": ids2, "attention_mask": am2}, task="detection", sep=1012)
    torch.save(dict(seed=17, keys=sorted(enc.state_dict().keys()), bert=dict(vocab=30522, hidden=64, layers=2, heads=4, inter=96, max_pos=512),
                    ids=ids, am=am, hidden_long=long["hidden"], ids2=ids2, am2=am2, hidden_short=short["hidden"]),
               os.path.join(OUT, "ref_bert_chunk.pt"))
    print("ref_bert_chunk.pt", tuple(long["hidden"].shape), int(am[0].sum()))


def gen_postproc():
    """The reference's own HIPIE_IMG.inference (NMS / flat top-100 / x4 upsample + threshold / class pooling / softmax(sigmoid/T) /
    semantic einsum / panoptic merge) and ddetrs.segmentation_postprocess, executed on synthetic head outputs with the REAL
    detectron2 Instances / Boxes classes.  Two variants: mean pooling + FG/BG class masking (training yaml) and max pooling +
    class-agnostic background (ADE eval yaml)."""
    hi = ref_import.ref("hipie_img")
    dd = ref_import.ref("models.ddetrs")
    boxes_mod = ref_import._load_file("detectron2.structures.boxes", f"{ref_import.REF_ROOT}/detectron2/structures/boxes.py")
    inst_mod = ref_import._load_file("detectron2.structures.instances", f"{ref_import.REF_ROOT}/detectron2/structures/instances.py")
    for m in (hi, dd):
        m.Instances, m.Boxes = inst_mod.Instances, boxes_mod.Boxes
    hi.retry_if_cuda_oom = lambda f: f
    g = torch.Generator().manual_seed(21)
    B, nbg, nfg, nmd, Lt, C, h, w = 2, 3, 40, 12, 24, 6, 16, 20
    H, W = 4 * h, 4 * w
    pos_map = {1: [1, 2], 2: [4], 3: [6, 7, 8], 4: [10], 5: [12, 13], 6: [15]}
    is_thing = {1: True, 2: True, 3: True, 4: True, 5: False, 6: False}
    out = {"pred_logits": torch.randn(B, nbg + nfg, Lt, generator=g) * 2 - 1, "pred_boxes": torch.rand(B, nbg + nfg, 4, generator=g) * 0.5 + 0.2,
           "pred_masks": torch.randn(B, nbg + nfg, 1, h, w, generator=g) * 3, "pred_boxious": torch.randn(B, nbg + nfg, 1, generator=g),
           "pred_logits_maskdino": torch.randn(B, nmd, Lt, generator=g) * 2 - 1, "pred_masks_maskdino": torch.randn(B, nmd, h, w, generator=g) * 3,
           "pred_boxes_maskdino": torch.rand(B, nmd, 4, generator=g)}
    out["pred_boxes"][:, 10:14] = out["pred_boxes"][:, 5:9] + 0.003            # near-duplicates so that NMS removes something

    def blobs(n):      # one soft rectangle per query (real mask logits are blob-like; pure noise never passes the overlap filter)
        m = torch.full((B, n, h, w), -6.0)
        for b in range(B):
            for q in range(n):
                y0, x0 = int(torch.randint(0, h - 5, (1,), generator=g)), int(torch.randint(0, w - 6, (1,), generator=g))
                m[b, q, y0:y0 + int(torch.randint(3, 6, (1,), generator=g)), x0:x0 + int(torch.randint(3, 7, (1,), generator=g))] = 6.0
        return m + torch.randn(B, n, h, w, generator=g)
    out["pred_masks"] = blobs(nbg + nfg).unsqueeze(2)
    out["pred_masks_maskdino"] = blobs(nmd)
    image_sizes = [(H, W), (H - 6, W - 10)]
    sizes = [(H, W), (50, 70)]                                                 # second image: resized semantic / panoptic output
    variants = {}
    for tag, max_pool, agn in (("mean_fgbg", False, False), ("maxpool_agnostic", True, True)):
        fake = types.SimpleNamespace(num_bg=nbg, num_fg=nfg, ota=True, mode_free_inference=False, max_pool_token_test=max_pool, enable_clip=False,
                                     demo_only=False, mask_on=True, mask_stride=4, mask_thres=0.5, use_bg_for_pano=False, bg_cls_agnostic=agn,
                                     transform_eval=True, pano_temp=0.06, object_mask_threshold=0.25, overlap_threshold=0.8,
                                     detr=types.SimpleNamespace(bg_query_from_lang=False, decouple_decoder=True, mask_dino_fixed_linear_head=False))
        fake.semantic_inference = lambda *a, f=fake: hi.HIPIE_IMG.semantic_inference(f, *a)
        fake.panoptic_inference = lambda *a, f=fake: hi.HIPIE_IMG.panoptic_inference(f, *a)
        with torch.no_grad():
            res = hi.HIPIE_IMG.inference(fake, out["pred_logits"].clone(), out["pred_boxes"].clone(), out["pred_masks"].clone(), image_sizes, pos_map, C,
                                         task="detection", iou_pred=out["pred_boxious"].clone(), is_thing=[is_thing, is_thing], sizes=sizes,
                                         output={k: v.clone() for k, v in out.items()})
        packed = []
        for r, (oh, ow) in zip(res, sizes):
            inst = r["instances"]
            raw_boxes = inst.pred_boxes.tensor.clone()        # segmentation_postprocess rescales the Boxes object in place
            post = dd.segmentation_postprocess(inst, oh, ow)
            packed.append(dict(pred_boxes=raw_boxes, scores=inst.scores, pred_classes=inst.pred_classes, pred_masks=inst.pred_masks,
                               post_boxes=post.pred_boxes.tensor, post_masks=post.pred_masks, post_scores=post.scores, post_classes=post.pred_classes,
                               sem_seg=r["sem_seg"], panoptic_seg=r["panoptic_seg"][0], segments_info=r["panoptic_seg"][1]))
        variants[tag] = dict(max_pool=max_pool, bg_cls_agnostic=agn, results=packed)
        print("ref_postproc", tag, [len(p["scores"]) for p in packed], [len(p["segments_info"]) for p in packed])
    g2 = dict(logits=torch.randn(2, 5, Lt, generator=g))
    g2["mean_fg"] = hi.convert_grounding_to_od_logits(g2["logits"], C, pos_map, is_thing=is_thing, mode="FG")
    g2["max_bg"] = hi.convert_grounding_to_od_logits(g2["logits"], C, pos_map, is_thing=is_thing, mode="BG", max_pool=True)
    torch.save(dict(out=out, image_sizes=image_sizes, sizes=sizes, pos_map=pos_map, is_thing=is_thing, num_classes=C, nbg=nbg, nfg=nfg,
                    variants=variants, pool=g2), os.path.join(OUT, "ref_postproc.pt"))


SYNTH_VOCAB = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", ".", ",", "(", ")", "-", "person", "traffic", "light", "fire", "hydrant", "teddy", "bear",
               "hair", "dr", "##ier", "tooth", "##brush", "sky", "other", "merged", "wall", "brick", "the", "man", "in", "red", "shirt", "left", "of",
               "dog", "skate", "##board", "a", "b", "##c", "tv", "potted", "plant", "cell", "phone", "wine", "glass"]


def synth_tokenizer(tmpdir):
    from transformers import BertTokenizerFast
    path = os.path.join(tmpdir, "vocab.txt")
    with open(path, "w") as f:
        f.write("\n".join(SYNTH_VOCAB) + "\n")
    tok = BertTokenizerFast(vocab={t: i for i, t in enumerate(SYNTH_VOCAB)}, do_lower_case=True)      # transformers 5.x signature
    assert tok.vocab_size == len(SYNTH_VOCAB) and tok("hair drier").input_ids == [2, 17, 18, 19, 3]
    return tok


def gen_prompts():
    """coco_dataset_mapper_uni.py create_queries_and_maps / create_positive_dict / clean_name with a BertTokenizerFast over a small
    synthetic vocabulary (multi-word names, word pieces, unknown words, parenthesised suffixes, underscores, stuff classes)."""
    import tempfile
    mp = ref_import.ref("data.coco_dataset_mapper_uni")
    cats = [{"name": "person"}, {"name": "traffic light"}, {"name": "fire hydrant"}, {"name": "teddy bear"}, {"name": "hair drier"},
            {"name": "toothbrush"}, {"name": "sky-other-merged", "isthing": 0}, {"name": "wall_brick", "isthing": 0},
            {"name": "skateboard (toy)"}, {"name": "zebra"}, {"name": "tv"}, {"name": "potted plant"}, {"name": "cell phone"},
            {"name": "wine glass"}]
    with tempfile.TemporaryDirectory() as d:
        tok = synth_tokenizer(d)
        q_all, m_all = mp.create_queries_and_maps(cats, tok)
        q_things, m_things = mp.create_queries_and_maps(cats, tok, things_only=True)
    torch.save(dict(vocab=SYNTH_VOCAB, cats=cats, query=q_all, pos_map=m_all, query_things=q_things, pos_map_things=m_things,
                    clean=[(n, mp.clean_name(n)) for n in ("wall_brick", "skateboard (toy)", "a  b", "x_(y)_z")]),
               os.path.join(OUT, "ref_prompts.pt"))
    print("ref_prompts.pt", q_all[:60], {k: m_all[k] for k in list(m_all)[:5]})


def gen_r50():
    """detectron2/modeling/backbone/resnet.py: BasicStem + ResNet.make_default_stages(50, FrozenBN, stride_in_1x1=False), the
    backbone of BASELINE configs[0] (training/r50.yaml: RESNETS.DEPTH 50, STRIDE_IN_1X1 False, OUT_FEATURES res3-res5)."""
    ref_import.install()
    import detectron2.modeling as d2m
    import detectron2.modeling.backbone.backbone as bbmod
    bbmod.Backbone = d2m.Backbone
    r = ref_import._load_file("detectron2.modeling.backbone.resnet", f"{ref_import.REF_ROOT}/detectron2/modeling/backbone/resnet.py")
    m = r.ResNet(r.BasicStem(3, 64, norm="FrozenBN"), r.ResNet.make_default_stages(50, norm="FrozenBN", stride_in_1x1=False),
                 out_features=["res3", "res4", "res5"])
    randomize_(m, 23).eval()
    x = torch.randn(2, 3, 96, 72, generator=torch.Generator().manual_seed(24))
    with torch.no_grad():
        out = m(x)
    sub = lambda t: t[:, ::8].contiguous()           # every 8th channel is enough to pin the arithmetic and keeps the fixture small
    torch.save(dict(seed=23, keys=sorted(m.state_dict().keys()), x=x, out={k: sub(v) for k, v in out.items()}), os.path.join(OUT, "ref_r50.pt"))
    print("ref_r50.pt", {k: tuple(v.shape) for k, v in out.items()})


def gen_maskclip():
    """open_vocab/clip.py: the UNMODIFIED MaskCLIP / ClipAdapter classes, constructed through a stub `open_clip` whose
    create_model_and_transforms returns hipie_oracle.clip.CLIP (the restated open_clip 2.0.2 model, tiny configuration) -- so the mask-token
    construction, the attention-mask layout, ln_post / proj on the mask tokens, the logit scale clamp and the synonym ensembling that run
    here are the reference's own lines.  get_clip_logits is the reference's HIPIE_IMG method, called on a stand-in `self`."""
    import torchvision.transforms as T
    from hipie_oracle import clip as oc
    ref_import.install()
    cfg = dict(oc.TINY)
    model = oc.init_clip_(oc.CLIP(cfg), seed=31)
    import open_clip                                   # the stub module
    size = cfg["image_size"]
    preprocess = T.Compose([T.Resize(size, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(size), (lambda im: im), (lambda im: im),
                            T.Normalize(oc.OPENAI_MEAN, oc.OPENAI_STD)])      # open_clip transform.py image_transform(is_train=False)
    open_clip.create_model_and_transforms = lambda *a, **k: (model, None, preprocess)
    open_clip.tokenize = lambda texts: oc.synth_clip_tokenize(texts, cfg["text_ctx"], cfg["vocab"])
    import detectron2.utils.comm as comm
    comm.get_local_rank, comm.synchronize = (lambda: 0), (lambda: None)
    rc = ref_import.ref("open_vocab.clip")
    hi = ref_import.ref("hipie_img")
    mc = rc.MaskCLIP(name="tiny")
    g = torch.Generator().manual_seed(32)
    Q, H, W = 7, 40, 60
    image = torch.rand(1, 3, H, W, generator=g)
    mask = torch.full((1, Q, H // 4, W // 4), -5.0)
    for q in range(Q):                                   # blob-like mask logits: most patches are masked out, different ones per query
        y0, x0 = int(torch.randint(0, H // 4 - 4, (1,), generator=g)), int(torch.randint(0, W // 4 - 5, (1,), generator=g))
        mask[0, q, y0:y0 + 4, x0:x0 + 5] = 5.0
    mask = mask + torch.randn(mask.shape, generator=g)
    test_labels = [{"id": 1, "name": "person,child,girl"}, {"id": 2, "name": "wall"}, {"id": 3, "name": "zebra,okapi"}, {"id": 4, "name": "sky"},
                   {"id": 5, "name": "traffic light,signal"}]
    train_labels = [{"id": 1, "name": "person,people"}, {"id": 2, "name": "sky,clouds"}, {"id": 3, "name": "traffic light"}]
    names = [x["name"].split(",") for x in test_labels]
    labels = hi.prompt_labels(names, "photo")                           # helper.py:112-130 (imported by hipie_img.py)
    flat = [t for ls in labels for t in ls]
    ids = open_clip.tokenize(flat)
    with torch.no_grad():
        text_embed, text_enc = mc._encode_text(ids)                      # ClipAdapter._encode_text :152-166
        text_embed2 = mc.build_text_embed(labels, always_cache=True)    # clip.py:29-73 through the stub tokenizer
        out = mc(image, mask, text_embed, labels)
        pred_open_prob = torch.softmax(torch.randn(Q, len(test_labels), generator=g) * 2, -1)
        fused = {}
        for mode in ("MUL", "ADD"):
            fake = types.SimpleNamespace(train_labels=train_labels, clip=mc, clip_agg_mode=mode)
            fused[mode] = hi.HIPIE_IMG.get_clip_logits(fake, 0, [test_labels], mask, types.SimpleNamespace(tensor=image), pred_open_prob,
                                                       alpha=0.35, beta=0.7)
        single = rc.MaskCLIP.pred_logits(mc, out["mask_embed"], text_embed[:1], [labels[0][:1]])       # one prompt: the sigmoid branch input
    assert torch.equal(text_embed, text_embed2)
    torch.save(dict(cfg=cfg, seed=31, image=image, mask=mask, ids=ids, labels=labels, test_labels=test_labels, train_labels=train_labels,
                    text_embed=text_embed, mask_embed=out["mask_embed"], logits=out["mask_pred_open_logits"], pred_open_prob=pred_open_prob,
                    fused=fused, single_logits=single, logit_scale=float(mc.logit_scale)), os.path.join(OUT, "ref_maskclip.pt"))
    print("ref_maskclip.pt", tuple(out["mask_embed"].shape), tuple(out["mask_pred_open_logits"].shape), {k: tuple(v.shape) for k, v in fused.items()})


CONFIGS = ["training/r50.yaml", "training/vit_huge_32g.yaml", "eval/image_joint_vit_huge_32g_pan_maskdino_ade_test.yaml"]


def gen_configs():
    """projects/HIPIE/configs: the YAMLs the config tests load, with every file their _BASE_ chains and MASKDINO.CONFIG_PATH
    reach, as parsed by yaml.safe_load and keyed by the path under the reference root, so that a test can lay the same tree out
    again and load it through hipie_b200.config."""
    import json
    import yaml
    cfg_root = "projects/HIPIE/configs"
    tree, todo = {}, [f"{cfg_root}/{c}" for c in CONFIGS]
    while todo:
        rel = os.path.normpath(todo.pop())
        if rel in tree:
            continue
        with open(os.path.join(ref_import.REF_ROOT, rel)) as f:
            d = tree[rel] = yaml.safe_load(f)
        if "_BASE_" in d:
            todo.append(os.path.join(os.path.dirname(rel), d["_BASE_"]))
        path = d.get("MODEL", {}).get("MASKDINO", {}).get("CONFIG_PATH")
        if path:
            todo.append(path)
    for d in tree.values():
        assert yaml.safe_load(yaml.safe_dump(d)) == d          # the test writes them back out with safe_dump
    with open(os.path.join(OUT, "ref_configs.json"), "w") as f:
        json.dump({"configs": CONFIGS, "root": cfg_root, "files": dict(sorted(tree.items()))}, f, indent=1)
        f.write("\n")
    print("ref_configs.json", sorted(tree))


def gen_msda_binding():
    """ops/functions/ms_deform_attn_func.py: the positional argument list MSDeformAttnFunction.forward passes to the pybind op
    `MultiScaleDeformableAttention.ms_deform_attn_forward` (recorded by a stand-in module), and ms_deform_attn_core_pytorch on the
    same seeded inputs."""
    seen = []
    msda = types.ModuleType("MultiScaleDeformableAttention")
    msda.ms_deform_attn_forward = lambda *args: seen.append(args) or torch.zeros(())
    prev, sys.modules["MultiScaleDeformableAttention"] = sys.modules.get("MultiScaleDeformableAttention"), msda
    f = ref_import._load_file("ref_ms_deform_attn_func", f"{ref_import.HIPIE}/models/deformable_detr/ops/functions/ms_deform_attn_func.py")
    sys.modules["MultiScaleDeformableAttention"] = prev
    g = torch.Generator().manual_seed(41)
    inputs = dict(value=torch.rand(1, 20, 2, 4, generator=g), shapes=torch.tensor([(4, 4), (2, 2)], dtype=torch.long),
                  level_start_index=torch.tensor([0, 16]), sampling_loc=torch.rand(1, 3, 2, 2, 2, 2, generator=g),
                  attn_weight=torch.rand(1, 3, 2, 2, 2, generator=g))
    im2col_step = 64
    with torch.no_grad():
        f.MSDeformAttnFunction.apply(*inputs.values(), im2col_step)
        core = f.ms_deform_attn_core_pytorch(inputs["value"], inputs["shapes"], inputs["sampling_loc"], inputs["attn_weight"])
    (args,) = seen
    call = [next(n for n, t in inputs.items() if a is t) if torch.is_tensor(a) else ("im2col_step" if a == im2col_step else None)
            for a in args]
    assert None not in call
    torch.save(dict(inputs=inputs, im2col_step=im2col_step, call=call, core=core), os.path.join(OUT, "ref_msda_binding.pt"))
    print("ref_msda_binding.pt", call, tuple(core.shape))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["vit", "transformer", "maskdino", "condinst", "bert", "postproc", "prompts", "r50", "maskclip", "configs",
                             "msda_binding"]
    for w in which:
        globals()["gen_" + w]()
