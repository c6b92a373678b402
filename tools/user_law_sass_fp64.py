"""FP64 instructions per chain x row of the user-law gradient sweeps, from cuobjdump -sass (no GPU
needed): the "lanes" kernel of the Poisson regression at P = D = 8 with the hand-written gradient
(tests/user_laws.py) and with forward-mode gradients (tests/user_laws_forward.py), compiled by NVRTC
with the library's options.  Prints the FP64 instructions of every loop of each kernel; the row loop
is unrolled 4 times (sweep_user.cuh), so per row = count / 4.  With --chunked P K: the "lanes" kernel
of every chunk of the forward-mode Poisson regression at P = D compiled at chunk width K (the
library's kernel extmcmc_user_lanes_f<K>c<c>), and the hand-written one at the same P.

    python tools/user_law_sass_fp64.py [--chunked P K]
"""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import user_laws as ul, user_laws_forward as uf
csrc = os.path.join(ROOT, 'extensiblemcmc.jl_b200', 'csrc')
TMP = tempfile.mkdtemp()
try:
    nv = C.CDLL("libnvrtc.so.12")
except OSError:
    nv = C.CDLL("/usr/local/cuda/lib64/libnvrtc.so.12")
def build(src, P, D, mode, K=None, c=0):
    hdr = ['sweep_user.cuh', 'dual.cuh', 'tma.cuh']
    law = {1: 'Law', 2: 'Law<extmcmc::Dual<EXTMCMC_P>>'}[mode] if K is None else f'Law<extmcmc::Dual<{K}>>'
    tail = f"{mode}" if K is None else f"{mode}, {K}, {c}"
    s = f"#define EXTMCMC_P {P}\n#define EXTMCMC_D {D}\n"
    s += "typedef signed char int8_t; typedef unsigned char uint8_t; typedef int int32_t; typedef unsigned int uint32_t;\ntypedef long long int64_t; typedef unsigned long long uint64_t;\n"
    s += src + '\n#include "sweep_user.cuh"\n'
    s += f'extern "C" __global__ void __launch_bounds__(128) k(extmcmc::UserSweepArgs a) {{ extmcmc::user_sweep<{law}, EXTMCMC_P, EXTMCMC_D, 1, 32, {tail}>(a); }}\n'
    prog = C.c_void_p()
    hs = (C.c_char_p * 3)(*[open(os.path.join(csrc, h), 'rb').read() for h in hdr])
    hn = (C.c_char_p * 3)(*[h.encode() for h in hdr])
    assert nv.nvrtcCreateProgram(C.byref(prog), s.encode(), b"u.cu", 3, hs, hn) == 0
    opts = [b"-arch=sm_100a", b"-std=c++17", b"-fmad=false"]
    rc = nv.nvrtcCompileProgram(prog, 3, (C.c_char_p * 3)(*opts))
    n = C.c_size_t(); nv.nvrtcGetProgramLogSize(prog, C.byref(n)); lg = C.create_string_buffer(n.value); nv.nvrtcGetProgramLog(prog, lg)
    assert rc == 0, lg.value.decode()
    nv.nvrtcGetCUBINSize(prog, C.byref(n)); buf = C.create_string_buffer(n.value); nv.nvrtcGetCUBIN(prog, buf)
    fn = os.path.join(TMP, f"m{mode}_{K}_{c}.cubin"); open(fn, 'wb').write(buf.raw)
    return subprocess.run(['cuobjdump', '-sass', fn], capture_output=True, text=True).stdout
FP64 = re.compile(r"\b(DADD|DMUL|DFMA|DSETP|DMNMX|DMMA|MUFU\.\w*64\w*|F2F\.F64\S*|DRND|F2I\.F64\S*|I2F\.F64\S*)\b")
def loops(sass):
    ins = []
    for line in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m: ins.append((int(m.group(1), 16), m.group(2)))
    out = []
    for a, t in ins:
        m = re.search(r"BRA\s+(?:`\(\.L_x_\d+\)\s*)?0x([0-9a-f]+)", t) or re.search(r"BRA .*?0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) < a:
            lo = int(m.group(1), 16)
            body = [x for b, x in ins if lo <= b <= a]
            out.append((lo, a, sum(1 for x in body if FP64.search(x)), len(body)))
    total = sum(1 for _, x in ins if FP64.search(x))
    return out, total
if len(sys.argv) == 4 and sys.argv[1] == "--chunked":
    P, K = int(sys.argv[2]), int(sys.argv[3])
    jobs = [("hand-written", ul.POISSON_REG, 1, None, 0)]
    jobs += [(f"forward chunk {c} of width {K}", uf.POISSON_REG, 2, K, c) for c in range(-(-P // K))]
else:
    P = 8
    jobs = [("hand-written", ul.POISSON_REG, 1, None, 0), ("forward", uf.POISSON_REG, 2, None, 0)]
for name, src, mode, K, c in jobs:
    sass = build(src, P, P, mode, K, c)
    lp, tot = loops(sass)
    print(name, "kernel FP64 total", tot)
    for l in lp: print("   loop %05x-%05x fp64 %d of %d instr" % l)
