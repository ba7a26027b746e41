"""CPU: the drop-in claim of INTEGRATION.md §1 against the REAL reference's detector, as recorded in
tests/golden/reference_detector.json by oracle/make_golden.py.  There the reference's own ``YoloXDetector`` was built around
``rvt_b200``'s backbone (``build_recurrent_backbone`` pointed at ``rvt_b200``), checked, and its model config, state_dict
layout (keys, shapes, dtypes), stage dims and strides recorded.  Here ``rvt_b200``'s detector, whose PAFPN / YOLOX head are
sized from our ``get_stage_dims`` / ``get_strides``, must reproduce that layout, and a checkpoint with the reference
detector's layout must load strictly into it and round-trip."""
import json
import os

import pytest
import torch

import rvt_b200
from rvt_b200.detection import YoloXDetector
from tests.golden_configs import DETECTOR_CASES

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_detector.json')


@pytest.fixture(scope='module')
def reference():
    with open(GOLDEN) as f:
        return json.load(f)


def _layout(sd):
    return {k: [list(v.shape), str(v.dtype).replace('torch.', '')] for k, v in sd.items()}


def _checkpoint(layout, seed):
    """seeded state_dict with the given layout (stands in for a reference checkpoint)"""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, (shape, dtype) in layout.items():
        dt = getattr(torch, dtype)
        sd[k] = (torch.randn(shape, generator=g).to(dt) if dt.is_floating_point else
                 torch.randint(0, 1000, tuple(shape), generator=g, dtype=dt))
    return sd


@pytest.mark.parametrize('embed_dim,dim_head', DETECTOR_CASES)       # RVT-B / S / T
def test_reference_detector_builds_around_our_backbone(reference, embed_dim, dim_head):
    ref = reference[f'{embed_dim}_{dim_head}']
    model = YoloXDetector(ref['model_cfg'])
    assert isinstance(model.backbone, rvt_b200.RNNDetector)
    # FPN / head were sized from our get_stage_dims / get_strides exactly as the reference sized them from its own backbone
    assert list(model.backbone.get_stage_dims((2, 3, 4))) == ref['stage_dims']
    assert list(model.backbone.get_strides((2, 3, 4))) == ref['strides']
    assert _layout(model.state_dict()) == ref['state_dict']
    # a reference checkpoint loads strictly (whole detector, Lightning strips the 'mdl.' prefix) and round-trips
    ckpt = _checkpoint(ref['state_dict'], embed_dim * 100 + dim_head)
    model.load_state_dict(ckpt, strict=True)
    for k, v in model.backbone.state_dict().items():
        assert torch.equal(v, ckpt['backbone.' + k]), k
    back = model.state_dict()
    assert back.keys() == ckpt.keys()
    for k, v in ckpt.items():
        assert torch.equal(back[k], v), k
