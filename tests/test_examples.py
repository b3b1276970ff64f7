"""The example scripts build their problem on the host and then call the device.  Without a CUDA device
they must stop at the first numerical step with the library's own error - there is no CPU fallback to
fall into - which also exercises all of their host code.  The device is hidden from a child process
(tests/nodevice.py), so these run on machines with a GPU too."""
import os

import pytest

from nodevice import run_without_device

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('script,argv', [('camcaldemo.py', []), ('prague2016_pm.py', ['s3']), ('ps_postproc.py', [])])
def test_examples_reach_the_device_call_and_fail_loudly_without_one(script, argv, tmp_path):
    err = run_without_device('''
import runpy
from dbat_b200._lib import DbatError
sys.argv = %r
try:
    runpy.run_path(%r, run_name='__main__')
    print(repr(None))
except DbatError as e:
    print(repr(str(e)))
''' % ([script] + argv, os.path.join(ROOT, 'examples', script)), cwd=tmp_path)
    assert err is not None and 'CUDA' in err


def test_script_runner_fails_loudly_without_a_device():
    raised = run_without_device('''
from dbat_b200 import rundbatscript
from dbat_b200._lib import DbatError
try:
    rundbatscript(%r, write=False)
    print(repr(False))
except DbatError:
    print(repr(True))
''' % os.path.join(ROOT, 'tests', 'golden', 'camcaldemo', 'camcaldemo.xml'))
    assert raised
