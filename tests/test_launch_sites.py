"""Every kernel of the library is launched through quip::launch (csrc/common.cuh), which counts the launch, opts into
dynamic shared memory, applies programmatic dependent launch and checks the arguments against the kernel's parameter
types.  A launch written any other way would skip one of those."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'quip_b200', 'csrc')
FORBIDDEN = {'<<<': '<<<', 'cudaFuncSetAttribute': r'\bcudaFuncSetAttribute\b',
             'cudaLaunchKernelEx': r'\bcudaLaunchKernelEx', 'void* args[]': r'void\s*\*\s*args\s*\[\s*\]'}
# api.cu holds the helper's attribute cache (raise_smem_limit)
ALLOWED = {'api.cu': {'cudaFuncSetAttribute'}}


def test_kernels_launch_only_through_the_helper():
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith('.cu'))
    assert 'qgemv.cu' in sources and 'api.cu' in sources
    found = []
    for name in sources:
        with open(os.path.join(CSRC, name)) as f:
            for i, line in enumerate(f, 1):
                found += [f'{name}:{i}: {line.strip()}' for what, pat in FORBIDDEN.items()
                          if what not in ALLOWED.get(name, ()) and re.search(pat, line)]
    assert not found, '\n'.join(found)
