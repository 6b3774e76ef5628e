"""from_reference_cfg(): snapshotting the reference's published configs (stored in tests/golden/reference_cfgs.json)
gives our named configs."""
from tests.helpers import load_reference_cfgs


def test_snapshot_matches_named_configs():
    from yolact_b200.config import CONFIGS, from_reference_cfg
    ref = load_reference_cfgs()
    assert sorted(ref) == sorted(CONFIGS)
    for name, mine in CONFIGS.items():
        snap = from_reference_cfg(ref[name])
        for key in ("backbone", "backbone_layers", "dcn_layers", "dcn_interval", "selected_layers", "max_size",
                    "pred_aspect_ratios", "use_square_anchors", "num_classes", "fpn_features", "use_maskiou",
                    "rescore_mask", "rescore_bbox", "nms_top_k", "nms_conf_thresh", "nms_thresh",
                    "max_num_detections", "normalize", "to_float"):
            assert getattr(snap, key) == getattr(mine, key), (name, key)
        for a, b in zip(snap.pred_scales, mine.pred_scales):
            assert [float(x) for x in a] == [float(x) for x in b], name
