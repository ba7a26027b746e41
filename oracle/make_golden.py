"""TEST INFRASTRUCTURE — run ONLY in the build container (needs /root/reference):

    python oracle/make_golden.py

1. imports the real reference (via oracle/_refshim.py), loads deterministic synthetic
   parameters into it (numpy RandomState seeds, oracle.backbone_oracle.synth_params);
2. checks oracle/backbone_oracle.py and oracle/voxel_oracle.py against it (asserts);
3. writes the REFERENCE's outputs to tests/golden/*.npz (small: strided subsamples +
   full-tensor sums for the big configs), so the GPU box — which has no /root/reference —
   can test both the oracle and the CUDA path against the reference.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import _refshim  # noqa: E402

_refshim.install()
from oracle import backbone_oracle as bo  # noqa: E402
from oracle import voxel_oracle as vo  # noqa: E402
from tests.golden_configs import (BACKBONE_CASES, MIXED_DENSITY_CASES, VOXEL_CASES, make_time_glitched, make_voxel_events,  # noqa: E402
                                  spec_of)
from oracle import neighbours_oracle as no  # noqa: E402
from oracle import detection_oracle as do  # noqa: E402
from tests.golden_configs import DETECTION_CASES, DETECTOR_CASES, POSTPROCESS_CASES, detection_inputs  # noqa: E402
from tests.helpers import GRAD_CASES, grad_sub, case_inputs, train_loss  # noqa: E402

from models.detection.recurrent_backbone import build_recurrent_backbone  # noqa: E402
from data.utils.representations import MixedDensityEventStack, StackedHistogram  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')


def ref_cfg(spec: bo.BackboneSpec):
    return _refshim.DictConfig(dict(
        name='MaxViTRNN', compile=dict(enable=False, args=dict(mode='reduce-overhead')),
        input_channels=spec.input_channels, enable_masking=spec.enable_masking,
        partition_split_32=1, embed_dim=spec.embed_dim, dim_multiplier=list(spec.dim_multiplier),
        num_blocks=list(spec.num_blocks), T_max_chrono_init=[4, 8, 16, 32],
        stem=dict(patch_size=spec.patch_size),
        stage=dict(downsample=dict(type='patch', overlap=spec.overlap, norm_affine=True),
                   attention=dict(use_torch_mha=False, partition_size=tuple(spec.partition_size),
                                  dim_head=spec.dim_head, attention_bias=True, mlp_activation='gelu',
                                  mlp_gated=False, mlp_bias=True, mlp_ratio=4, drop_mlp=0, drop_path=0,
                                  ls_init_value=spec.ls_init_value, norm_eps=spec.norm_eps),
                   lstm=dict(dws_conv=spec.dws_conv, dws_conv_only_hidden=spec.dws_conv_only_hidden,
                             dws_conv_kernel_size=spec.dws_conv_kernel_size, drop_cell_update=0))))


def sub(t: torch.Tensor, stride: int) -> np.ndarray:
    return t.contiguous().reshape(-1)[::stride].numpy().copy()


def run_backbone_case(name, case):
    spec = spec_of(case)
    torch.manual_seed(0)
    ref = build_recurrent_backbone(ref_cfg(spec)).eval()
    params = bo.synth_params(spec, case['seed'], case.get('gamma_mode', 'uniform'))
    ref_keys = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert ref_keys == bo.param_shapes(spec), 'oracle.param_shapes disagrees with the reference'
    ref.load_state_dict(params, strict=True)
    b, h, w, L = case['batch'], case['height'], case['width'], case['steps']
    stride = case.get('sub', 1)
    out = {}
    r_states, o_states = None, None
    worst = 0.0
    with torch.no_grad():
        for step in range(L):
            x = bo.synth_events_tensor(case['seed'] * 1000 + step, b, spec.input_channels, h, w).float()
            mask = None
            if spec.enable_masking:
                rs = np.random.RandomState(case['seed'] + 77 + step)
                mask = torch.from_numpy(rs.uniform(size=(b, h // 4, w // 4)) < 0.2)
            r_out, r_states = ref(x, r_states, mask)
            o_out, o_states = bo.backbone_forward(x, o_states, params, spec, mask)
            if case.get('reset_at') == step:       # harness-style in-place reset of sample 0
                for (hh, cc) in r_states:
                    hh[0] = 0
                    cc[0] = 0
                for (hh, cc) in o_states:
                    hh[0] = 0
                    cc[0] = 0
            for s in range(4):
                for a, bb in ((r_out[s + 1], o_out[s + 1]), (r_states[s][0], o_states[s][0]),
                              (r_states[s][1], o_states[s][1])):
                    worst = max(worst, float((a - bb).abs().max()))
            if step in case.get('save_steps', [L - 1]):
                for s in range(4):
                    hh, cc = r_states[s]
                    out[f'step{step}_h{s}'] = sub(hh, stride)
                    out[f'step{step}_c{s}'] = sub(cc, stride)
                    out[f'step{step}_h{s}_sum'] = np.float64(hh.double().sum().item())
                    out[f'step{step}_c{s}_sum'] = np.float64(cc.double().sum().item())
                    out[f'step{step}_h{s}_abssum'] = np.float64(hh.double().abs().sum().item())
    assert worst < 2e-5, (name, worst)
    np.savez_compressed(os.path.join(GOLD, f'backbone_{name}.npz'), **out)
    print(f'backbone {name}: oracle-vs-reference max abs diff {worst:.2e}; '
          f'{sum(v.size for v in out.values())} values saved')


def run_backbone_grad_case(name, steps):
    """Training-step pin: gradients of tests.helpers.train_loss over `steps` unrolled timesteps (states carried,
    modules/detection.py:150-199) from the REFERENCE under autograd, fp32 CPU; the oracle must agree."""
    case = BACKBONE_CASES[name]
    spec = spec_of(case)
    torch.manual_seed(0)
    ref = build_recurrent_backbone(ref_cfg(spec)).train()
    params = bo.synth_params(spec, case['seed'], case.get('gamma_mode', 'uniform'))
    ref.load_state_dict(params, strict=True)
    xs = case_inputs(case, steps)
    outs, st = [], None
    for x in xs:
        o, st = ref(x.float(), st, None)
        outs.append(o)
    loss_r = train_loss(outs, st)
    loss_r.backward()
    g_ref = {k: p.grad.detach().clone() for k, p in ref.named_parameters()}
    po = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    outs, st = [], None
    for x in xs:
        o, st = bo.backbone_forward(x.float(), st, po, spec)
        outs.append(o)
    loss_o = train_loss(outs, st)
    loss_o.backward()
    worst = 0.0
    for k, g in g_ref.items():
        e = float((po[k].grad - g).norm() / g.norm().clamp_min(1e-12))
        worst = max(worst, e)
    assert worst < 1e-4 and abs(float(loss_o.detach()) - float(loss_r.detach())) <= 1e-5 * abs(float(loss_r.detach())), (name, worst)
    out = {'loss': np.float64(float(loss_r))}
    for k, g in g_ref.items():
        out['g.' + k] = sub(g, grad_sub(name))
        out['n.' + k] = np.float64(g.double().norm().item())
    np.savez_compressed(os.path.join(GOLD, f'backbone_grads_{name}.npz'), **out)
    print(f'backbone grads {name}: oracle-vs-reference worst rel-L2 {worst:.2e}; loss {float(loss_r):.6f}; '
          f'{sum(v.size for v in out.values())} values saved')


def run_voxel_case(name, case):
    x, y, p, t = make_voxel_events(case)
    out = {}
    for fast in (True, False):
        sh = StackedHistogram(case['bins'], case['height'], case['width'], case.get('cutoff', 10), fast)
        ref = sh.construct(*(torch.from_numpy(a) for a in (x, y, p, t))).numpy()
        mine = vo.stacked_histogram(x, y, p, t, case['bins'], case['height'], case['width'],
                                    case.get('cutoff', 10), fast)
        assert ref.dtype == np.uint8 and ref.shape == (2 * case['bins'], case['height'], case['width'])
        assert np.array_equal(ref, mine), name
        out['fast' if fast else 'slow'] = ref
    np.savez_compressed(os.path.join(GOLD, f'voxel_{name}.npz'), **out)
    print(f'voxel {name}: bit-exact; n={len(x)} max={out["fast"].max()}')


def _reference_function(path, name, extra_globals):
    """Pull ONE function out of a reference source file that cannot be imported as a module here (its imports need h5py /
    hdf5plugin) and compile it as is -- decorators dropped (numba's @jit is an optimisation, not semantics)."""
    import ast
    src = open(path).read()
    tree = ast.parse(src)
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == name:
            node.decorator_list = []
            mod = ast.Module(body=[node], type_ignores=[])
            ns = dict(extra_globals)
            exec(compile(ast.fix_missing_locations(mod), path, 'exec'), ns)
            return ns[name]
    raise KeyError(name)


def run_detection_cases():
    """SURVEY 8 f2: oracle.detection_oracle vs the reference's YOLOPAFPN / YOLOXHead / postprocess; the REFERENCE's outputs
    are committed (tests/golden/det.npz)."""
    from models.detection.yolox_extension.models.yolo_pafpn import YOLOPAFPN
    from models.detection.yolox.models.yolo_head import YOLOXHead
    from models.detection.yolox.utils.boxes import postprocess
    out = {}
    for name, c in DETECTION_CASES.items():
        torch.manual_seed(0)
        fpn = YOLOPAFPN(depth=c['depth'], in_stages=(2, 3, 4), in_channels=c['in_channels']).eval()
        head = YOLOXHead(num_classes=c['num_classes'], strides=(8, 16, 32), in_channels=c['in_channels']).eval()
        sd_f = do.synth_state({k: tuple(v.shape) for k, v in fpn.state_dict().items()}, c['seed'])
        sd_h = do.synth_state({k: tuple(v.shape) for k, v in head.state_dict().items()}, c['seed'] + 1)
        fpn.load_state_dict(sd_f, strict=True)
        head.load_state_dict(sd_h, strict=True)
        feats = {k: torch.from_numpy(v) for k, v in detection_inputs(c).items()}
        with torch.no_grad():
            r = fpn(feats)
            ro, losses = head(r)
            o = do.pafpn_forward(feats, sd_f, depth=c['depth'])
            oo = do.head_forward(o, sd_h)
        assert losses is None
        w1 = max(float((a - b).abs().max()) for a, b in zip(r, o))
        w2 = float(((ro - oo).abs() / ro.abs().clamp_min(1.0)).max())
        assert w1 < 1e-5 and w2 < 1e-5, (name, w1, w2)
        for i, t in enumerate(r):
            out[f'{name}_fpn{i}'] = t.numpy()
        out[f'{name}_head'] = ro.numpy()
        print(f'detection {name}: oracle-vs-reference fpn {w1:.1e}, head {w2:.1e}; head out {tuple(ro.shape)}')
    for name, c in POSTPROCESS_CASES.items():
        pred = do.synth_predictions(c['seed'], c['batch'], c['anchors'], c['num_classes'])
        ref = postprocess(torch.from_numpy(pred.copy()), c['num_classes'], c['conf'], c['nms'])
        mine = do.postprocess(pred, c['num_classes'], c['conf'], c['nms'])
        for i, (a, b) in enumerate(zip(ref, mine)):
            assert (a is None) == (b is None), name
            if a is not None:
                assert a.shape == b.shape and np.array_equal(a.numpy(), b), (name, i)
                out[f'{name}_img{i}'] = a.numpy()
            else:
                out[f'{name}_img{i}'] = np.zeros((0, 7), np.float32)
        print(f'postprocess {name}: oracle == reference (torchvision batched_nms), {[0 if a is None else len(a) for a in ref]} detections')
    np.savez_compressed(os.path.join(GOLD, 'det.npz'), **out)


def state_layout(sd):
    """{key: [shape, dtype name]} of a state_dict"""
    return {k: [list(v.shape), str(v.dtype).replace('torch.', '')] for k, v in sd.items()}


def run_reference_detector_cases():
    """INTEGRATION.md section 1: the reference's own YoloXDetector built around rvt_b200's backbone (its PAFPN / YOLOX head
    sized from our get_stage_dims / get_strides) has the reference detector's state_dict, and checkpoints load strictly both
    ways.  The model config, the reference detector's state_dict layout, stage dims and strides go to
    tests/golden/reference_detector.json (tests/test_reference_integration_cpu.py)."""
    import json
    import yaml
    import models.detection.yolox_extension.models.detector as det
    import rvt_b200
    out = {}
    for embed_dim, dim_head in DETECTOR_CASES:
        with open(os.path.join(_refshim.REFERENCE_ROOT, 'config', 'model', 'maxvit_yolox', 'default.yaml')) as f:
            cfg = yaml.safe_load(f)['model']
        cfg['backbone']['embed_dim'] = embed_dim
        cfg['backbone']['stage']['attention']['dim_head'] = dim_head
        cfg['backbone']['stage']['attention']['partition_size'] = [6, 10]    # what config/modifier.py:36-41 derives for 1Mpx
        cfg['backbone']['stage']['attention']['ls_init_value'] = 1e-5        # (PyYAML reads the literal 1e-5 as a string)
        cfg['backbone']['in_res_hw'] = [384, 640]
        cfg['head']['num_classes'] = 3
        ref_model = det.YoloXDetector(_refshim.DictConfig(cfg))
        ref_builder = det.build_recurrent_backbone
        det.build_recurrent_backbone = rvt_b200.build_recurrent_backbone
        try:
            our_model = det.YoloXDetector(_refshim.DictConfig(cfg))             # reference FPN + head around rvt_b200.RNNDetector
        finally:
            det.build_recurrent_backbone = ref_builder
        assert isinstance(our_model.backbone, rvt_b200.RNNDetector)
        layout = state_layout(ref_model.state_dict())
        assert state_layout(our_model.state_dict()) == layout
        our_model.load_state_dict(ref_model.state_dict(), strict=True)
        ref_model.load_state_dict(our_model.state_dict(), strict=True)
        dims, strides = ref_model.backbone.get_stage_dims((2, 3, 4)), ref_model.backbone.get_strides((2, 3, 4))
        assert our_model.backbone.get_stage_dims((2, 3, 4)) == dims and our_model.backbone.get_strides((2, 3, 4)) == strides
        out[f'{embed_dim}_{dim_head}'] = dict(model_cfg=cfg, state_dict=layout, stage_dims=list(dims), strides=list(strides))
        print(f'detector {embed_dim}/{dim_head}: reference detector around rvt_b200 backbone matches, {len(layout)} entries')
    with open(os.path.join(GOLD, 'reference_detector.json'), 'w') as f:
        json.dump(out, f, sort_keys=True)
        f.write('\n')


def run_neighbour_cases():
    """SURVEY 8 f4: oracle.neighbours_oracle vs the reference's own code; the REFERENCE's outputs go to tests/golden/neigh.npz"""
    out = {}
    pre = '/root/reference/scripts/genx/preprocess_dataset.py'
    ref_downsample = _reference_function(pre, 'downsample_ev_repr', {'torch': torch})
    ref_correct_time = _reference_function(pre, '_correct_time', {'np': np})
    # downsample_ev_repr on a StackedHistogram output (uint8) and on a MixedDensity output (int8)
    c = VOXEL_CASES['uniform']
    x, y, p, t = make_voxel_events(c)
    sh = StackedHistogram(c['bins'], c['height'], c['width'], 10, True).construct(*(torch.from_numpy(a) for a in (x, y, p, t)))
    ds = ref_downsample(sh.unsqueeze(0), 0.5)[0].numpy()
    assert np.array_equal(ds, no.downsample_ev_repr(sh.numpy())), 'downsample_ev_repr (uint8)'
    out['ds_u8'] = ds
    odd = torch.from_numpy(np.random.RandomState(3).randint(0, 255, (3, 37, 51)).astype(np.uint8))     # odd H, W
    ds_odd = ref_downsample(odd.unsqueeze(0), 0.5)[0].numpy()
    assert np.array_equal(ds_odd, no.downsample_ev_repr(odd.numpy())), 'downsample_ev_repr (odd sizes)'
    out['ds_odd_in'], out['ds_odd'] = odd.numpy(), ds_odd
    # _correct_time
    tg = make_time_glitched(31, 20000)
    tr = tg.copy()
    ref_correct_time(tr)
    assert np.array_equal(tr, no.correct_time(tg)), '_correct_time'
    out['ct'] = tr
    # window indices: the reference's expression IS np.searchsorted (:511-516); pin the two branches
    ts = np.sort(np.random.RandomState(32).randint(0, 2_000_000, 50000).astype(np.int64))
    q = np.arange(50_000, 2_000_000, 50_000, dtype=np.int64)
    s_d, e_d = no.event_window_indices(ts, q, None, 50)
    s_n, e_n = no.event_window_indices(ts, q, 3000, None)
    assert np.array_equal(e_d, np.searchsorted(ts, q, side='right')) and np.array_equal(s_d, np.searchsorted(ts, q - 50000, side='left'))
    out['win_start_dt'], out['win_end'], out['win_start_n'] = s_d, e_d, s_n
    # MixedDensityEventStack
    for name, c in MIXED_DENSITY_CASES.items():
        x, y, p, t = make_voxel_events(c)
        ref = MixedDensityEventStack(c['bins'], c['height'], c['width'], c['cutoff']).construct(
            *(torch.from_numpy(a) for a in (x, y, p, t))).numpy()
        mine = no.mixed_density_stack(x, y, p, t, c['bins'], c['height'], c['width'], c['cutoff'])
        assert ref.dtype == np.int8 and np.array_equal(ref, mine), name
        out[name] = ref
        print(f'mixed density {name}: bit-exact; n={len(x)} range [{ref.min()}, {ref.max()}]')
    np.savez_compressed(os.path.join(GOLD, 'neigh.npz'), **out)
    print('neighbours: downsample / correct_time / window indices / mixed density pinned to the reference')


if __name__ == '__main__':
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    only = [a.split('=', 1)[1] for a in sys.argv if a.startswith('--only=')]     # --only=<case>[,<case>...]
    only = set(only[0].split(',')) if only else None
    want = lambda n: only is None or n in only
    if '--grads-only' not in sys.argv and want('neigh'):
        run_neighbour_cases()
    if '--grads-only' not in sys.argv and want('det'):
        run_detection_cases()
    if '--grads-only' not in sys.argv and want('reference_detector'):
        run_reference_detector_cases()
    if '--grads-only' not in sys.argv:
        for n, c in VOXEL_CASES.items():
            if want(n):
                run_voxel_case(n, c)
    if '--grads-only' not in sys.argv:
        for n, c in BACKBONE_CASES.items():
            if want(n):
                run_backbone_case(n, c)
    for n, steps in GRAD_CASES.items():
        if want(n) and '--no-grads' not in sys.argv:
            run_backbone_grad_case(n, steps)
