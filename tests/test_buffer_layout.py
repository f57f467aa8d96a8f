"""CPU: the layout of the reduction buffers red32 / red64 / gsum / scal as include/oriana_b200.h states it (the ORI_R64_*,
ORI_GSUM_* and ORI_SC_* slots and the size macros), against its mirror in oriana_b200/_lib.py and the buffers that
problem.gene_buffers allocates.  The header's values come from the C compiler itself."""
import os
import re
import subprocess

import pytest

from oriana_b200 import _lib
from oriana_b200.problem import gene_buffers, pad_k

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'oriana_b200.h')
SLOTS = re.findall(r'^#define (ORI_(?:R64|GSUM|SC)_[A-Z_]+) ', open(HEADER).read(), flags=re.M)


@pytest.fixture(scope='module')
def header(tmp_path_factory):
    """Runs a C program built against the header: no arguments prints every slot constant, `p KP third` the three
    buffer sizes."""
    d = tmp_path_factory.mktemp('layout')
    src = d / 'layout.c'
    src.write_text('#include <stdio.h>\n#include <stdlib.h>\n#include "oriana_b200.h"\n'
                   'int main(int argc, char** argv) {\n'
                   '    if (argc == 4) {\n'
                   '        const int p = atoi(argv[1]), KP = atoi(argv[2]), third = atoi(argv[3]);\n'
                   '        printf("%lld %lld %lld\\n", (long long)ORI_RED32_FLOATS(p, KP, third),\n'
                   '               (long long)ORI_RED64_DOUBLES(p, KP), (long long)ORI_GSUM_DOUBLES(KP));\n'
                   '        return 0;\n'
                   '    }\n'
                   + ''.join('    printf("%s %%d\\n", (int)(%s));\n' % (s, s) for s in SLOTS) +
                   '    return 0;\n}\n')
    exe = d / 'layout'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-I', os.path.dirname(HEADER),
                    str(src), '-o', str(exe)], check=True)
    return lambda *args: subprocess.run([str(exe), *map(str, args)], check=True, capture_output=True, text=True).stdout


def test_python_mirrors_every_slot_of_the_header(header):
    assert {'ORI_R64_NSLOTS', 'ORI_GSUM_NSLOTS', 'ORI_SC_NSLOTS', 'ORI_SC_ELBO_LAST', 'ORI_SC_ITER'} <= set(SLOTS)
    values = dict(line.split() for line in header().splitlines())
    assert {name: int(v) for name, v in values.items()} == {name: getattr(_lib, name) for name in SLOTS}
    # the slot names the Python side uses are exactly the header's
    assert sorted(n for n in dir(_lib) if re.match(r'ORI_(R64|GSUM|SC)_', n) and not callable(getattr(_lib, n))) == sorted(SLOTS)


# K in {1, 10, 40}: the CUDA-core KP of each K and the tensor path's KPs (32, 64) that hold it
CASES = [(K, KP) for K in (1, 10, 40) for KP in sorted({pad_k(K), 32, 64}) if KP >= K]


@pytest.mark.parametrize('sparse', [False, True])
@pytest.mark.parametrize('K, KP', CASES)
def test_gene_buffers_have_the_header_sizes(header, K, KP, sparse):
    p = 977
    red32, red64, gsum = (int(v) for v in header(p, KP, int(sparse)).split())
    assert (_lib.ORI_RED32_FLOATS(p, KP, sparse), _lib.ORI_RED64_DOUBLES(p, KP), _lib.ORI_GSUM_DOUBLES(KP)) == (red32, red64, gsum)
    g = gene_buffers(p, K, KP, 'cpu', dropout=not sparse, sparse=sparse, trace_cap=3)
    assert g['red32'].numel() == red32 and g['red32'].shape == (red32 // (p * KP), p, KP)
    assert g['red64'].shape == (red64,) and g['gsum'].shape == (gsum,)
    assert g['scal'].shape == (_lib.ORI_SC_NSLOTS,)
