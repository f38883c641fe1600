"""CPU: the reference's UNMODIFIED Hydra YAMLs (its configs/model tree, stored under tests/golden/reference_configs) resolve
to this repo's drop-in classes and construct the full SamPt object tree (SURVEY §8b boundary contract)."""
import os

import pytest
import torch

REF_CFG = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs")


def test_reference_yaml_instantiates_dropin(tmp_path):
    from oracle import pips_ref
    from sampt_b200 import hydra_lite, synth
    pips_sd = synth.condition_pips(synth.make_state_dict(pips_ref.pips_state_dict_shapes(), 1))
    ckpt = synth.write_pips_checkpoint_dir(pips_sd, str(tmp_path / "models" / "pips_ckpts" / "reference_model"))
    cfg = hydra_lite.compose_model(REF_CFG, {
        "point_tracker": "pips", "sam@sam_predictor.sam_model": "sam_vit_base",
        "sam_predictor._target_": "segment_anything.predictor.SamPredictor",   # docs/04-running-experiments.md:56-58
        "sam_predictor.sam_model.checkpoint": None,
        "positive_points_per_mask": 4, "negative_points_per_mask": 0,
    }, cwd=str(tmp_path))
    assert cfg["_target_"] == "sam_pt.modeling.sam_pt.SamPt"
    assert cfg["point_tracker"]["checkpoint_path"] == ckpt
    assert cfg["sam_predictor"]["sam_model"]["image_encoder"]["embed_dim"] == 768
    assert cfg["sam_predictor"]["sam_model"]["image_encoder"]["out_chans"] == 256  # ${ ..prompt_embed_dim }
    assert cfg["sam_predictor"]["sam_model"]["mask_decoder"]["transformer"]["embedding_dim"] == 256  # ${ ...prompt_embed_dim }
    model = hydra_lite.instantiate(cfg)
    import sam_pt.modeling.sam_pt as m
    assert type(model) is m.SamPt
    assert model.positive_points_per_mask == 4 and model.iterative_refinement_iterations == 12
    assert model.sam_predictor.model.image_encoder.depth == 12
    assert model.sam_predictor.model.image_encoder.global_attn_indexes == (2, 5, 8, 11)
    assert hasattr(model.sam_predictor, "set_image") and hasattr(model.sam_predictor, "predict_torch")
    # the reference's error behaviour at the boundary
    model.train()
    with pytest.raises(NotImplementedError):
        model({"image": [torch.zeros((3, 8, 8), dtype=torch.uint8)], "target_hw": (8, 8)})


def test_vit_huge_override_composes():
    from sampt_b200 import hydra_lite
    cfg = hydra_lite.compose_model(REF_CFG, {"point_tracker": "pips", "sam@sam_predictor.sam_model": "sam_vit_huge"}, cwd="/x")
    enc = cfg["sam_predictor"]["sam_model"]["image_encoder"]
    assert (enc["depth"], enc["embed_dim"], enc["num_heads"]) == (32, 1280, 16)
    assert enc["global_attn_indexes"] == [7, 15, 23, 31]
    assert cfg["sam_predictor"]["sam_model"]["checkpoint"] == "/x/models/sam_ckpts/sam_vit_h_4b8939.pth"


def test_default_hq_config_instantiates(tmp_path):
    """configs/model/sam_pt.yaml's own defaults select HQ-SAM ViT-H + `segment_anything_hq.predictor.SamPredictor`
    (sam_pt.yaml:3-8); only the tracker group is switched to PIPS here; the no-override default is covered below."""
    from oracle import pips_ref
    from sampt_b200 import hydra_lite, synth
    pips_sd = synth.condition_pips(synth.make_state_dict(pips_ref.pips_state_dict_shapes(), 1))
    synth.write_pips_checkpoint_dir(pips_sd, str(tmp_path / "models" / "pips_ckpts" / "reference_model"))
    cfg = hydra_lite.compose_model(REF_CFG, {"point_tracker": "pips", "sam_predictor.sam_model.checkpoint": None,
                                             # keep the unit test small: shrink the ViT, everything else as configured
                                             "sam_predictor.sam_model.image_encoder.depth": 2,
                                             "sam_predictor.sam_model.image_encoder.global_attn_indexes": [1]}, cwd=str(tmp_path))
    assert cfg["sam_predictor"]["_target_"] == "segment_anything_hq.predictor.SamPredictor"
    assert cfg["sam_predictor"]["sam_model"]["_target_"] == "sam_pt.modeling.sam.SamHQHydra"
    assert cfg["sam_predictor"]["sam_model"]["mask_decoder"]["_target_"] == "segment_anything_hq.modeling.mask_decoder_hq.MaskDecoderHQ"
    assert cfg["sam_predictor"]["sam_model"]["mask_decoder"]["vit_dim"] == 1280  # ${..image_encoder.embed_dim}
    model = hydra_lite.instantiate(cfg)
    import segment_anything_hq.predictor as hp
    assert type(model.sam_predictor) is hp.SamPredictor
    assert "mask_decoder.hf_token.weight" in model.sam_predictor.model.state_dict()


def test_default_cotracker_config_instantiates(tmp_path):
    """configs/model/sam_pt.yaml with NO tracker override: the reference's default point tracker is CoTracker
    (sam_pt.yaml:3, configs/model/point_tracker/cotracker.yaml); a checkpoint written with upstream's key names loads."""
    from oracle import cotracker_ref
    from sampt_b200 import hydra_lite, synth
    sd = synth.condition_cotracker(synth.make_state_dict(cotracker_ref.cotracker_state_dict_shapes(), 3))
    ck = tmp_path / "models" / "cotracker_ckpts"
    ck.mkdir(parents=True)
    torch.save({"model": sd}, str(ck / "cotracker_stride_4_wind_8.pth"))
    cfg = hydra_lite.compose_model(REF_CFG, {"sam_predictor.sam_model.checkpoint": None,
                                             "sam_predictor.sam_model.image_encoder.depth": 2,
                                             "sam_predictor.sam_model.image_encoder.global_attn_indexes": [1]}, cwd=str(tmp_path))
    pt = cfg["point_tracker"]
    assert pt["_target_"] == "sam_pt.point_tracker.cotracker.CoTrackerPointTracker"
    assert pt["interp_shape"] == [384, 512] and pt["visibility_threshold"] == 0.7
    assert pt["support_grid_size"] == 2 and pt["support_grid_every_n_frames"] == 12
    model = hydra_lite.instantiate(cfg)
    from sam_pt.point_tracker.cotracker import CoTrackerPointTracker
    assert type(model.point_tracker) is CoTrackerPointTracker
    got = model.point_tracker.model.state_dict()
    assert set(got) == set(sd)
    k = "updateformer.space_blocks.5.attn.qkv.weight"
    assert torch.equal(got[k].cpu(), sd[k])
