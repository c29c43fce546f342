"""Every compiled lidar kernel variant against the oracle, at every fixed-point width, and the device EDT at its limits.

launch_lidar picks one of 80 instantiations: lidar_kernel and lidar_maps_kernel <FB, COUNT, MODE> with FB = 19..22 (the
tuned variants) or 0 (generic).  The runs below use thin synthetic maps at both ends of every width from 24 down to 17
fraction bits (tests/helpers.py SYNTH_MAPS), map sets at every common width, and handles that force the generic variant at
tuned widths.  Each run is one reset step, noise-free, and must equal the oracle bit for bit:
scans_f64, scans_f32, the observation's lidar channel, terminated and, with lookup counting, the lookup count.  The one
exception are the beams an opponent lowers (A = 2): they end on the post kernel's ray / edge intersection, not on the lidar
kernel's march, and are held to 4 ulp.  Every run also checks which variant ran (f110_get_lidar_variant), and the union of
the variants must be all 80.
"""
import math
import os

import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

B = 1080
LEAN = ('obs', 'reward', 'terminated')
# (agents, outputs) -> the mode launch_lidar must select with noise_std = 0 and no host noise
MODES = {1: (1, None), 2: (1, LEAN), 0: (2, None), 3: (2, LEAN + ('scans_f32',))}
SETS = {   # map sets: every slot gets poses
    'set19': ('w19_8190', 'w21_1500'), 'set20': ('w20_4094', 'w22_511'), 'set21': ('w21_1500', 'w24_200'),
    'set22': ('w22_1022', 'w23_254', 'w22_511'), 'set23': ('w23_254', 'w24_200'), 'set18': ('w18_8191', 'w24_200'),
}


def _poses(name, A):
    p = H.synthetic_poses(name)
    if A == 1:
        return p[:, None, :]
    # the opponent 0.6 m ahead of the ego along its heading: the opponent ray cast lowers some beams
    q = p.copy()
    q[:, 0] += 0.6 * np.cos(p[:, 2]); q[:, 1] += 0.6 * np.sin(p[:, 2])
    return np.stack([p, q], 1)


_ORACLE = {}


def _oracle(name, A, eps=1e-4, max_range=30.0):
    key = (name, A, eps, max_range)
    if key not in _ORACLE:
        from oracle.f110_oracle import Oracle
        _, dt, res, origin = H.synthetic_map(name)
        poses = _poses(name, A)
        o = Oracle(len(poses), A, eps=eps, max_range=max_range)
        o.set_map_arrays(dt, res, origin)
        out = o.reset(poses)
        ref = dict(scans=out['scans'].copy(), obs=out['obs'].copy(), terminated=out['terminated'].copy(),
                   lookups=int(o.last_lookups))
        # the beams the opponent ray-cast lowered: there the scan is not the lidar kernel's march but the post kernel's
        # ray / edge intersection (see _run)
        wall = np.stack([[o.scan(p)[0] for p in env] for env in poses])
        ref['lowered'] = ref['scans'].view(np.int64) != wall.view(np.int64)
        _ORACLE[key] = ref
    return _ORACLE[key]


def _run(maps, mode, count, narrow=False, eps=1e-4, max_range=30.0, image=False):
    """One reset step of a fresh handle holding `maps` (one name, or a set) -> (variant, list of mismatches)."""
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    A, outputs = MODES[mode]
    names = list(maps)
    refs = [_oracle(n, A, eps, max_range) for n in names]
    poses = np.concatenate([_poses(n, A) for n in names])
    slots = np.concatenate([np.full(len(r['terminated']), k, np.int32) for k, r in enumerate(refs)])
    sim = BatchSim(len(poses), A, outputs=outputs or ALL_OUTPUTS, noise_std=0.0, count_lookups=count,
                   narrow_fraction=narrow, eps=eps, max_range=max_range, device=0)
    bad = []
    try:
        if len(names) > 1:
            sim.set_maps([H.synthetic_map(n)[1:] for n in names])
            sim.set_env_maps(slots)
        elif image:
            free, dt, res, origin = H.synthetic_map(names[0])
            sim.set_map_image(free, res, origin)
            if not np.array_equal(sim.get_map().view(np.int64), dt.view(np.int64)):
                bad.append('device EDT differs from scipy')
        else:
            sim.set_map_arrays(*H.synthetic_map(names[0])[1:])
        look0 = sim.lookup_count()[0] if count else 0
        out = sim.reset(poses)
        torch.cuda.synchronize()
        variant = sim.lidar_variant()
        got = {k: v.cpu().numpy() for k, v in out.items()}
        want_scans = np.concatenate([r['scans'] for r in refs])
        lowered = np.concatenate([r['lowered'] for r in refs])
        lm = np.float32(30.0)
        want_obs = np.clip(np.nan_to_num(want_scans[:, 0].astype(np.float32)), 0, lm) / lm
        for name, g, w, low in (('scans_f64', got.get('scans_f64'), want_scans, lowered),
                                ('scans_f32', got.get('scans_f32'), want_scans.astype(np.float32), lowered),
                                ('obs lidar', got['obs'][:, :B], want_obs, lowered[:, 0]),
                                ("obs lidar (oracle's observation)", got['obs'][:, :B],
                                 np.concatenate([r['obs'] for r in refs])[:, :B], lowered[:, 0])):
            if g is None:
                continue
            # every beam the lidar kernel decides: bit for bit
            d = (g != w) & ~low
            if d.any():
                bad.append('%s: %d beams differ, first %s, max |d| %.3g' % (
                    name, d.sum(), np.argwhere(d)[:3].tolist(), np.abs(np.where(d, g - w, 0)).max()))
            # a beam an opponent lowers ends on the post kernel's ray / edge intersection, whose beam direction comes from
            # CUDA's double sincos and the oracle's from libm's cos / sin: the two may differ in the last bit
            d = (np.abs(g - w) > 4 * np.spacing(w)) & low
            if d.any():
                bad.append('%s: %d beams an opponent lowers differ by more than 4 ulp, first %s' % (
                    name, d.sum(), np.argwhere(d)[:3].tolist()))
        if not np.array_equal(got['terminated'], np.concatenate([r['terminated'] for r in refs])):
            bad.append('terminated differs')
        if count:
            # both count every distance-transform read of the reference's march, the first included; the kernel's
            # pipelined extra load and a redone ray's abandoned fast march are not counted
            look = sim.lookup_count()[0] - look0
            if look != sum(r['lookups'] for r in refs):
                bad.append('lookups %d != oracle %d' % (look, sum(r['lookups'] for r in refs)))
    finally:
        sim.close()
    return variant, bad


def _expected(maps, mode, count, narrow=False, eps=1e-4, max_range=30.0):
    fb = H.fraction_bits(max(max(H.synthetic_map(n)[0].shape) for n in maps))
    min_positive = min(H.synthetic_map(n)[2] for n in maps)       # one cell from an obstacle
    tuned = not narrow and max_range == 30.0 and 0 < eps < min_positive and 19 <= fb <= 22
    return dict(fraction_bits=fb, template_fb=fb if tuned else 0, mode=mode, maps=int(len(maps) > 1))


def _key(v, count):
    return ('lidar_maps_kernel' if v['maps'] else 'lidar_kernel', v['template_fb'], count, v['mode'])


ALL_VARIANTS = {(k, fb, c, m) for k in ('lidar_kernel', 'lidar_maps_kernel') for fb in (0, 19, 20, 21, 22)
                for c in (False, True) for m in range(4)}


def _plan():
    runs = []
    for mode in (1, 2, 0, 3):
        for count in (False, True):
            runs += [((n,), mode, count, {}) for n in sorted(H.SYNTH_MAPS)]
            runs += [(SETS[s], mode, count, {}) for s in sorted(SETS)]
    for kw in (dict(narrow=True), dict(max_range=25.0), dict(eps=0.05)):       # eps = the smallest positive cell of these
        runs += [(('w21_1500',), 1, True, kw), (('w20_4094',), 0, False, kw), (SETS['set20'], 3, True, kw)]
    runs.append((('w17_16383',), 1, True, dict(image=True)))     # a width-17 map built by the device EDT
    return runs


def test_yaws_are_libm_exact():
    for y in H.SYNTH_YAWS:
        assert np.cos(y) == math.cos(y) and np.sin(y) == math.sin(y), y


def test_every_variant_against_the_oracle():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    failures, seen, rows = [], {}, []
    for maps, mode, count, kw in _plan():
        variant, bad = _run(maps, mode, count, **kw)
        want = _expected(maps, mode, count, **{k: v for k, v in kw.items() if k != 'image'})
        if variant != want:
            bad.append('variant %s, expected %s' % (variant, want))
        label = '%s mode %d count %d %s' % ('+'.join(maps), mode, count, kw or '')
        if bad:
            failures.append((label, bad))
        seen.setdefault(_key(variant, count), label)
    missing = ALL_VARIANTS - set(seen)
    print('\n%-18s %3s %5s %4s  first run' % ('kernel', 'FB', 'COUNT', 'MODE'))
    for k in sorted(seen):
        print('%-18s %3d %5d %4d  %s' % (*k, seen[k]))
    print('%d of %d variants ran' % (len(set(seen) & ALL_VARIANTS), len(ALL_VARIANTS)))
    for label, msgs in failures:
        print('FAILED', label, msgs)
    assert not failures, failures
    assert not missing, sorted(missing, key=str)
    assert set(seen) == ALL_VARIANTS


# ---------------------------------------------------------------- the device EDT at its limits

def _edt_check(free, res=0.05, wide=False):
    """set_map_image on `free` (the narrow or, with wide=True, the general form) must give res * scipy's EDT bit for bit."""
    import torch
    from scipy.ndimage import distance_transform_edt
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    want = res * distance_transform_edt(np.where(free, 255., 0.))
    if wide:
        os.environ['F110_EDT_WIDE'] = '1'
    sim = BatchSim(1, 1, noise_std=0.0, device=0)
    try:
        sim.set_map_image(free, res, (0.0, 0.0, 0.0))
        got = sim.get_map()
    finally:
        os.environ.pop('F110_EDT_WIDE', None)
        sim.close()
    d = got != want
    assert not d.any(), (free.shape, wide, int(d.sum()), np.argwhere(d)[:3].tolist())


@pytest.mark.parametrize('shape', [(16, 32750), (32750, 16), (16, 32751), (32751, 16)])
def test_device_edt_at_the_narrow_forms_limit(shape):
    """H + W + 1 = 32767 is the largest map the 16-bit form takes; 32768 selects the general form.  One obstacle in a
    corner: the envelope's integers come closest to their 31-bit bound, and all but one row or column hold no obstacle."""
    free = np.ones(shape, bool)
    free[-1, -1] = False
    _edt_check(free)


@pytest.mark.parametrize('wide', [False, True])
@pytest.mark.parametrize('shape', [(1, 1), (1, 6), (6, 1), (3, 4), (70, 130), (130, 70), (200, 1030)])
def test_device_edt_without_obstacles(shape, wide):
    """scipy measures an obstacle-free mask from a virtual obstacle at (-1, 0): res * sqrt((r + 1)^2 + c^2)."""
    _edt_check(np.ones(shape, bool), res=0.07, wide=wide)
