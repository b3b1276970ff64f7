"""The C-ABI library builds for sm_100a, loads, and exports every symbol include/dbat_gpu.h
declares.  No compute calls here (no GPU in the build container)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_graft_build_and_exports(built_lib):
    import ctypes
    from dbat_b200 import _lib
    assert os.path.exists(built_lib)
    hdr = open(os.path.join(ROOT, 'include', 'dbat_gpu.h')).read()
    declared = set(re.findall(r'\b(dbat_[a-z_0-9]+)\s*\(', hdr))
    declared -= {'dbat_handle'}
    L = ctypes.CDLL(built_lib)
    for name in sorted(declared):
        assert hasattr(L, name), 'missing export ' + name
    assert declared == set(_lib.EXPORTS)


def test_struct_layouts_match_header():
    """ctypes mirrors of dbat_problem_desc / dbat_opts / dbat_result have the C sizes."""
    import subprocess
    import tempfile
    from dbat_b200 import _lib
    import ctypes
    src = '#include <stdio.h>\n#include "dbat_gpu.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n", sizeof(dbat_problem_desc), sizeof(dbat_opts), sizeof(dbat_result), sizeof(dbat_fwi_desc), sizeof(dbat_resect_desc));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, 't.c')
        open(c, 'w').write(src)
        exe = os.path.join(d, 't')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', exe])
        sizes = [int(v) for v in subprocess.check_output([exe]).split()]
    assert sizes == [ctypes.sizeof(_lib.ProblemDesc), ctypes.sizeof(_lib.Opts), ctypes.sizeof(_lib.Result),
                     ctypes.sizeof(_lib.FwiDesc), ctypes.sizeof(_lib.ResectDesc)]


def test_no_cpu_fallback_without_device(built_lib):
    """Without a CUDA device the product path fails loudly instead of computing on the CPU (device hidden from a
    child process, so this runs on machines with a GPU too)."""
    from nodevice import run_without_device
    raised = run_without_device('''
import dbat_b200
from dbat_b200.synth import make_scene
s, _ = make_scene(6, 30, rays=4, seed=1)
try:
    dbat_b200.Problem(s)
    print(repr(False))
except dbat_b200._lib.DbatError:
    print(repr(True))
''')
    assert raised


def test_product_does_not_import_oracle():
    import glob
    for f in glob.glob(os.path.join(ROOT, 'dbat_b200', '**', '*.py'), recursive=True):
        txt = open(f).read()
        assert not re.search(r'^\s*(from|import)\s+oracle', txt, re.M), f


def test_bench_reference_arm_runs_without_gpu():
    """`bench.py --impl reference` (the oracle port of the reference CPU algorithm on a bounded sample)
    must work on a box without CUDA and print one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '0',
                          '--nimg', '60', '--nop', '6000'],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'lm_iterations_per_s' and line['value'] > 0
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['value'] == line['value']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert line['gpu_launches'] == 0 and 'workload' in line['config'] and line['config']['same_config'] is True
    assert line['steps'] == 2
