"""Schur-phase time of projects with wide points (estimated points with more than 20 rays), A/B of library builds on
one B200:

    python tools/long_ray_bench.py base=variants/libdbatgpu_base.so new=dbat_b200/libdbatgpu.so > long_ray_bench.jsonl

Scenes: spread-long (tests/test_ray_spread.py: 160 images, 20 000 points, 817 of them wide) and the camcal demo.
For every scene, five rounds; every round runs each build in turn (alternating), on a fresh handle: three warm-up
steps, then 20 damped steps from the start vector, each one's `build_schur` phase (S assembly + Schur reduction,
Problem.phase_times) recorded.  A round's figure is the median over its steps; the result is the median over the
rounds and their spread.  Also prints the sizes of the wide-point index and staging buffers (schur_wide.cu), computed
from the scene, and the card.  One JSON line per (scene, build) on stdout; the card goes to stderr.
"""
import copy
import json
import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

ROUNDS, WARMUP, STEPS = 5, 3, 20
NSLOT, SSPART = 14, 16


def wide_bytes(s):
    """Bytes of the wide-point index (ints) and staging (doubles) that dbat_create allocates for scene s."""
    img, op = np.asarray(s.IP.img), np.asarray(s.IP.op)
    nImg, nOP = s.EO.val.shape[1], s.OP.val.shape[1]
    rays = np.bincount(op, minlength=nOP)
    wide = np.flatnonzero(s.bundle.est.OP.any(axis=0) & (rays > 20))
    nBig, nWObs = len(wide), int(rays[wide].sum())
    iswide = np.zeros(nOP, bool)
    iswide[wide] = True
    lists = {}
    for i, j in zip(img[iswide[op]], op[iswide[op]]):
        lists.setdefault(j, []).append(i)
    pairs = set()
    for l in lists.values():
        for a in l:
            for b in l:
                if a >= b:
                    pairs.add((a, b))
    index = 4 * (nWObs + (nImg + 1) + 2 * nWObs + 2 * len(pairs))
    staging = 8 * (18 * nWObs + 48 * nBig + 256 * ((nBig + SSPART - 1) // SSPART) + NSLOT * (NSLOT + 1))
    return dict(nBig=nBig, nWObs=nWObs, nWPair=len(pairs), index_bytes=index, staging_bytes=staging)


def scenes():
    from camcal_fixture import camcal_struct
    from oracle.dbatstruct import buildserialindices
    from test_ray_spread import scene
    c = camcal_struct()
    buildserialindices(c)
    return {'spread-long': scene('spread-long')[0], 'camcal': c}


def schur_ms(s):
    import dbat_b200
    x0 = dbat_b200.serialize(s)
    P = dbat_b200.Problem(s)
    for _ in range(WARMUP):
        P.normal_step(x0, 0.0, False)
    ms = []
    for _ in range(STEPS):
        P.normal_step(x0, 0.0, False)
        ms.append(P.phase_times()['build_schur'][0])
    P.close()
    return float(np.median(ms))


def main():
    from dbat_b200 import _lib
    builds = []
    for spec in sys.argv[1:]:
        name, path = spec.split('=', 1)
        dst = '/tmp/lrb_%s.so' % name
        shutil.copyfile(os.path.join(ROOT, path), dst)
        builds.append((name, dst))
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                          capture_output=True, text=True).stdout.strip()
    print('card:', card, file=sys.stderr)
    for sname, s in scenes().items():
        sizes = wide_bytes(s)
        times = {name: [] for name, _ in builds}
        for _ in range(ROUNDS):
            for name, path in builds:
                _lib._lib = None
                _lib.LIB_PATH = path
                times[name].append(schur_ms(copy.deepcopy(s)))
        for name, _ in builds:
            t = times[name]
            d = dict(scene=sname, build=name, schur_ms_median=float(np.median(t)), schur_ms_min=min(t), schur_ms_max=max(t),
                     rounds=t, card=card, **sizes)
            print(json.dumps(d), flush=True)


if __name__ == '__main__':
    main()
