import sys, ctypes as C, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import bls_ref as B
import lighthouse_b200
from lighthouse_b200 import bls
lighthouse_b200.init(0)
L = C.CDLL('tests/hostsim/libhostsim.so')
u = B.hash_to_field_fp2(bytes(range(32)))[0]
ub = u[0].to_bytes(48,'big')+u[1].to_bytes(48,'big')
o = C.create_string_buffer(16*96); L.hs_sswu_trace(ub, o)
rc, d = bls.debug_stage(8, ub, 16*96)
names = 'tv1 tv2 x1n x1d N D a na|t1 s|inv_na target y0 invD y1 x1 x y'.split()
for k in range(16):
    h, g = o.raw[96*k:96*k+96], d[96*k:96*k+96]
    print(names[k], 'OK' if h==g else 'DIFF c0 %s c1 %s' % (h[:48]==g[:48], h[48:]==g[48:]))
