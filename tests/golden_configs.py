"""Golden-fixture case table shared by oracle/make_golden.py (which mints tests/golden/*.npz
from the real reference) and the tests (which replay the same seeded inputs)."""
import numpy as np

from oracle import backbone_oracle as bo
from oracle import voxel_oracle as vo

# partition_size = (H/32, W/32) * 1/partition_split_32  (config/modifier.py:36-41)
BACKBONE_CASES = {
    # tiny, every stage small; P=6 (exercises heavy window padding 6->64)
    'tiny_p6': dict(embed_dim=32, dim_head=32, height=64, width=96, partition=(2, 3), batch=2,
                    steps=3, seed=11, save_steps=[0, 2]),
    # RVT-S style head dim 24, P=20
    'small_dh24': dict(embed_dim=48, dim_head=24, height=128, width=160, partition=(4, 5), batch=1,
                       steps=2, seed=12),
    # depthwise 3x3 on the hidden state only (reference default when dws_conv=True)
    'dws_hidden': dict(embed_dim=32, dim_head=32, height=64, width=96, partition=(2, 3), batch=2,
                       steps=3, seed=13, dws_conv=True, dws_only_hidden=True, reset_at=1),
    # depthwise 3x3 on cat(x, h)
    'dws_xh': dict(embed_dim=32, dim_head=32, height=64, width=96, partition=(2, 3), batch=1,
                   steps=2, seed=14, dws_conv=True, dws_only_hidden=False),
    # reference-default LayerScale init 1e-5 (SURVEY D10) + token masking in stage 1
    'ls_init_mask': dict(embed_dim=32, dim_head=32, height=64, width=96, partition=(2, 3), batch=2,
                         steps=2, seed=15, gamma_mode='init', enable_masking=True),
    # BASELINE configs[0]: RVT-Tiny Gen1 256x320 (P=80), bs 1, seq_len 5
    'rvt_t_gen1': dict(embed_dim=32, dim_head=32, height=256, width=320, partition=(8, 10), batch=1,
                       steps=5, seed=16, sub=7),
    # RVT-Base 1Mpx 384x640 (P=60), bs 1, 2 steps
    'rvt_b_1mpx': dict(embed_dim=64, dim_head=32, height=384, width=640, partition=(6, 10), batch=1,
                       steps=2, seed=17, sub=13),
    # BASELINE configs[1] shape: RVT-Base 1Mpx, bs 8, seq_len 21 (state drift over a whole benchmark sequence, SURVEY D11)
    'rvt_b_1mpx_bs8_l21': dict(embed_dim=64, dim_head=32, height=384, width=640, partition=(6, 10), batch=8,
                               steps=21, seed=18, sub=997, save_steps=[0, 10, 20], heavy=True),
    # BASELINE configs[3] shape: RVT-Small Gen1 256x320: dim_head 24 (padded head) WITH P = 80 (one window per 128-row tile)
    'rvt_s_gen1': dict(embed_dim=48, dim_head=24, height=256, width=320, partition=(8, 10), batch=2,
                       steps=3, seed=19, sub=11),
    # BASELINE configs[2] per-GPU shape: RVT-Base 1Mpx bs 3 (gradient golden, tests.helpers.GRAD_CASES)
    'rvt_b_1mpx_bs3': dict(embed_dim=64, dim_head=32, height=384, width=640, partition=(6, 10), batch=3,
                           steps=2, seed=20, sub=211, heavy=True),
}


def spec_of(case) -> bo.BackboneSpec:
    return bo.BackboneSpec(embed_dim=case['embed_dim'], dim_head=case['dim_head'],
                           partition_size=tuple(case['partition']),
                           dws_conv=case.get('dws_conv', False),
                           dws_conv_only_hidden=case.get('dws_only_hidden', True),
                           enable_masking=case.get('enable_masking', False))


VOXEL_CASES = {
    'uniform': dict(n=200000, height=72, width=128, bins=10, seed=1),
    'hot': dict(n=300000, height=48, width=64, bins=10, seed=2, hot_fraction=0.3, hot_pixels=2),
    'single': dict(n=1, height=10, width=12, bins=10, seed=3),
    'same_ts': dict(n=1000, height=16, width=16, bins=10, seed=4, same_timestamp=True),
    'empty': dict(n=0, height=8, width=8, bins=10, seed=5),
    'bins3_cut255': dict(n=100000, height=20, width=24, bins=3, seed=6, cutoff=None,
                         hot_fraction=0.5, hot_pixels=1),
    'big_t': dict(n=50000, height=32, width=32, bins=10, seed=7, t_offset=1 << 40, t_span=(1 << 31) + 12345),
}


def make_voxel_events(case):
    n = case['n']
    if n == 0:
        z = np.zeros(0, np.int64)
        return z, z.copy(), z.copy(), z.copy()
    x, y, p, t = vo.synth_events(case['seed'], n, case['height'], case['width'],
                                 t_span=case.get('t_span', 50000),
                                 hot_fraction=case.get('hot_fraction', 0.0),
                                 hot_pixels=case.get('hot_pixels', 16))
    if case.get('same_timestamp'):
        t = np.full(n, 12345, np.int64)
    t = t + np.int64(case.get('t_offset', 0))
    return x, y, p, t


# ---- SURVEY 8 f4: neighbours of the voxelizer -------------------------------------------------------------------
MIXED_DENSITY_CASES = {
    'md_uniform': dict(n=120000, height=48, width=64, bins=10, seed=21, cutoff=None),
    'md_hot_cut3': dict(n=150000, height=24, width=32, bins=10, seed=22, cutoff=3, hot_fraction=0.4, hot_pixels=2),
    'md_wrap': dict(n=60000, height=4, width=4, bins=4, seed=23, cutoff=None, hot_fraction=0.9, hot_pixels=1),   # int8 wrap-around
    'md_single': dict(n=1, height=6, width=8, bins=10, seed=24, cutoff=5),
    'md_same_ts': dict(n=2000, height=8, width=8, bins=10, seed=25, cutoff=None, same_timestamp=True),
    'md_empty': dict(n=0, height=8, width=8, bins=10, seed=26, cutoff=None),
    'md_bins1': dict(n=5000, height=8, width=8, bins=1, seed=27, cutoff=7),
}


def make_time_glitched(seed: int, n: int):
    """sorted timestamps with backwards glitches (what H5Reader._correct_time repairs)"""
    rs = np.random.RandomState(seed)
    t = np.sort(rs.randint(0, 1_000_000, n).astype(np.int64))
    bad = rs.uniform(size=n) < 0.02
    t = np.where(bad, t - rs.randint(1, 5000, n), t)
    t[0] = abs(t[0])
    return np.where(t < 0, 0, t)


# ---- SURVEY 8 f2: PAFPN + YOLOX head + postprocess ----------------------------------------------------------------
DETECTION_CASES = {
    # RVT-Base gen4 (1Mpx): stages 2-4 dims (128, 256, 512), depth 0.67, 3 classes; small spatial sizes
    'det_b_gen4': dict(in_channels=(128, 256, 512), depth=0.67, num_classes=3, batch=2, hw8=(12, 20), seed=51),
    # RVT-Tiny gen1: dims (64, 128, 256), depth 0.33, 2 classes
    'det_t_gen1': dict(in_channels=(64, 128, 256), depth=0.33, num_classes=2, batch=1, hw8=(16, 20), seed=52),
}
POSTPROCESS_CASES = {
    'pp_gen4': dict(seed=5, batch=3, anchors=5040, num_classes=3, conf=0.1, nms=0.45),
    'pp_small': dict(seed=6, batch=2, anchors=300, num_classes=2, conf=0.3, nms=0.45),
}
# whole detector (backbone + PAFPN + YOLOX head) at 1Mpx: (embed_dim, dim_head) of RVT-B / S / T
DETECTOR_CASES = [(64, 32), (48, 24), (32, 32)]


def detection_inputs(case):
    rs = np.random.RandomState(case['seed'] + 100)
    h, w = case['hw8']
    b = case['batch']
    return {st: (rs.normal(0, 0.3, (b, c, h >> i, w >> i))).astype(np.float32)
            for i, (st, c) in enumerate(zip((2, 3, 4), case['in_channels']))}
