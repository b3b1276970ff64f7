"""mex/dbat_mex.c - the MEX gateway a DBAT maintainer compiles (INTEGRATION.md) - compiled against a stand-in for
MATLAB's MEX API (tests/mexstub), linked to libdbatgpu.so and driven through its mexFunction entry.

CPU part: the gateway compiles warning-free, validates its arguments with the reference's error-id convention
(icpc_mex.c:499-577: mexErrMsgIdAndTxt("DBAT:<fn>:<id>", ...)) and maps a library failure (no CUDA device here) to
DBAT:dbat_mex:create with the library's own message.  GPU part: a whole session through the gateway."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tests'))


@pytest.fixture(scope='module')
def mex(built_lib, tmp_path_factory):
    import mexharness
    return mexharness.Harness(mexharness.build(tmp_path_factory.mktemp('mex'), built_lib))


def _scene():
    from dbat_b200.dbatstruct import buildserialindices
    from dbat_b200.synth import make_scene
    s, _ = make_scene(6, 30, rays=4, seed=1)
    if s.bundle.serial is None:
        buildserialindices(s)
    return s


def test_gateway_compiles_and_validates_its_arguments(mex):
    import mexharness
    E = mexharness.MexError
    with pytest.raises(E) as e:
        mex.call()
    assert e.value.id == 'DBAT:dbat_mex:nrhs'
    with pytest.raises(E) as e:
        mex.call(3.0)                                   # first argument is not a command string
    assert e.value.id == 'DBAT:dbat_mex:nrhs'
    with pytest.raises(E) as e:
        mex.call('create', 1.0)                         # not a struct
    assert e.value.id == 'DBAT:dbat_mex:nrhs'
    with pytest.raises(E) as e:
        mex.call('eval')                                # handle missing
    assert e.value.id == 'DBAT:dbat_mex:nrhs' and 'Handle' in e.value.msg
    with pytest.raises(E) as e:
        mex.call('eval', 1.0)                           # handle of the wrong class
    assert e.value.id == 'DBAT:dbat_mex:badHandle'
    d = mexharness.desc_struct(_scene())
    bad = dict(d); del bad['EOval']
    with pytest.raises(E) as e:
        mex.call('create', bad)
    assert e.value.id == 'DBAT:dbat_mex:badField' and e.value.msg == 'EOval'
    bad = dict(d); bad['OPval'] = d['OPval'][:-1]
    with pytest.raises(E) as e:
        mex.call('create', bad)
    assert e.value.id == 'DBAT:dbat_mex:badSize' and e.value.msg == 'OPval'
    bad = dict(d); bad['IPimg'] = d['IPimg'].astype(np.float64)       # indices must arrive as int64
    with pytest.raises(E) as e:
        mex.call('create', bad)
    assert e.value.id == 'DBAT:dbat_mex:badField' and e.value.msg == 'IPimg'
    with pytest.raises(E) as e:
        mex.call('forwintersect', 1.0)
    assert e.value.id == 'DBAT:dbat_mex:nrhs'
    assert mex.H.hs_lock_count() == 0 and mex.H.hs_has_at_exit() == 1


def test_gateway_reports_the_library_error_without_a_device(mex):
    """No CPU fallback behind the gateway either: create fails with the library's message (the same harness in a
    child process with the device hidden, so this runs on machines with a GPU too)."""
    from nodevice import run_without_device
    ident, msg, locks = run_without_device('''
import mexharness
from test_mex_gateway import _scene
mex = mexharness.Harness(%r)
try:
    mex.call('create', mexharness.desc_struct(_scene()))
    print(repr((None, None, mex.H.hs_lock_count())))
except mexharness.MexError as e:
    print(repr((e.id, e.msg, mex.H.hs_lock_count())))
''' % mex.H._name)
    assert ident == 'DBAT:dbat_mex:create' and 'code -' in msg
    assert locks == 0                                  # nothing stays locked after a failed create


@pytest.mark.gpu
def test_session_through_the_gateway_matches_the_ctypes_path():
    """create / eval / jacobian / solve / cov / covstats / forwintersect / destroy through mexFunction against the
    same calls through dbat_b200 (own process: a marshalling bug must not take the test session down)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'mex_worker.py')], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode == 0 and 'MEX SESSION OK' in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
