"""Builds the in-tree CUDA library (sm_100a only) with nvcc.  No JIT cache: the .so lives next
to the sources so it travels with the repo snapshot to the GPU box."""
import hashlib
import os
import subprocess
import sys

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc')
LIB = os.path.join(CSRC, 'libautoml_b200.so')
STAMP = LIB + '.stamp'
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
    '-Xcompiler', '-fPIC', '--shared',
]


def _sources():
  return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest():
  h = hashlib.sha256()
  inc = os.path.join(os.path.dirname(os.path.dirname(CSRC)), 'include', 'automl_b200.h')
  headers = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh'))
  for f in _sources() + headers + [inc]:
    with open(f, 'rb') as fh:
      h.update(os.path.basename(f).encode())   # not the absolute path: the tree may be moved after the build
      h.update(fh.read())
  h.update(' '.join(FLAGS).encode())
  return h.hexdigest()


def build(force=False, verbose=False):
  """Compiles every .cu under csrc/ into libautoml_b200.so (skipped when up to date)."""
  digest = _digest()
  if not force and os.path.exists(LIB) and os.path.exists(STAMP):
    with open(STAMP) as f:
      if f.read().strip() == digest:
        return LIB
  if not os.path.exists(NVCC):
    raise RuntimeError('nvcc not found at %s and %s is stale/missing' % (NVCC, LIB))
  cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + _sources() + ['-o', LIB]
  res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  if verbose or res.returncode != 0:
    sys.stderr.write(res.stdout)
  if res.returncode != 0:
    raise RuntimeError('nvcc failed (%d)' % res.returncode)
  with open(STAMP, 'w') as f:
    f.write(digest)
  return LIB


if __name__ == '__main__':
  print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
