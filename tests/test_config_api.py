"""CPU: the reference's own YAMLs (tests/golden/ref_configs.json, laid out by the `ref_configs` fixture) load unchanged through
the config surface."""
import os

import pytest


@pytest.mark.parametrize("rel", ["training/r50.yaml", "training/vit_huge_32g.yaml",
                                 "eval/image_joint_vit_huge_32g_pan_maskdino_ade_test.yaml"])
def test_reference_yaml_loads(rel, ref_configs):
    from hipie_b200.config import setup_cfg
    from hipie_b200.modeling.hipie_img import hp_from_cfg
    cfg = setup_cfg(os.path.join(ref_configs, rel), ["MODEL.DEVICE", "cuda"])
    assert cfg.MODEL.META_ARCHITECTURE == "HIPIE_IMG"
    assert cfg.MODEL.DDETRS.TWO_STAGE_NUM_PROPOSALS == 900 and cfg.MODEL.DDETRS.TWO_STAGE_NUM_BG_PROPOSALS == 10
    assert cfg.MODEL.MASKDINO.ENABLED is True
    assert cfg._maskdino_cfg is not None and cfg._maskdino_cfg.MODEL.MaskDINO.DEC_LAYERS == 9
    hp = hp_from_cfg(cfg)
    assert hp["md_queries"] == 300 and hp["md_dim_ff"] == 2048
    if "vit" in rel:
        assert hp["backbone"] == "vit" and hp["vit"]["embed_dim"] == 1280 and hp["vit"]["depth"] == 32
    else:
        assert hp["backbone"] == "r50"
    assert hp["max_query_len"] in (512, 4096)


def test_cfg_node_semantics(tmp_path):
    from hipie_b200.config import CfgNode, get_cfg
    base = tmp_path / "base.yaml"
    child = tmp_path / "child.yaml"
    base.write_text("MODEL:\n  WEIGHTS: a\n  RESNETS:\n    DEPTH: 50\nINPUT:\n  MIN_SIZE_TRAIN: (1024,)\n")
    child.write_text("_BASE_: base.yaml\nMODEL:\n  WEIGHTS: b\n")
    cfg = get_cfg()
    cfg.merge_from_file(str(child))
    assert cfg.MODEL.WEIGHTS == "b" and cfg.MODEL.RESNETS.DEPTH == 50 and cfg.INPUT.MIN_SIZE_TRAIN == (1024,)
    cfg.merge_from_list(["MODEL.RESNETS.DEPTH", "101", "MODEL.MASK_ON", "on"])
    assert cfg.MODEL.RESNETS.DEPTH == 101 and cfg.MODEL.MASK_ON is True
    c2 = cfg.clone()
    c2.MODEL.WEIGHTS = "c"
    assert cfg.MODEL.WEIGHTS == "b"
    cfg.freeze()
    with pytest.raises(AttributeError):
        cfg.MODEL.WEIGHTS = "z"


def test_registry_and_no_cpu_path():
    from hipie_b200.registry import META_ARCH_REGISTRY, _register_defaults
    _register_defaults()
    cls = META_ARCH_REGISTRY.get("HIPIE_IMG")
    with pytest.raises(RuntimeError):
        cls(hp=dict(backbone="vit"), device="cpu")
