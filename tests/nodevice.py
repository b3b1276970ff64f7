"""Run a snippet in a child Python with every CUDA device hidden (CUDA_VISIBLE_DEVICES empty), so that the behaviour
without a device is tested on machines with a GPU as well.  Test infrastructure only."""
import ast
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_without_device(code, cwd=None):
    """Runs `code` (which must print the repr of a Python literal as its last line) and returns that literal."""
    head = 'import sys\nsys.path[:0] = [%r, %r]\n' % (ROOT, os.path.join(ROOT, 'tests'))
    r = subprocess.run([sys.executable, '-c', head + code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=600, cwd=cwd)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return ast.literal_eval(r.stdout.strip().splitlines()[-1])
