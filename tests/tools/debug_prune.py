import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from pclean_b200.host_fixture import model as M
from tests.test_engine_parity import _setup_synth
cfg = M.InferenceConfig(1, 20)
out = {}
for prune in (1, 0):
    model, query, ir, dirty, truth, o, e = _setup_synth(cfg, n_rows=6000, H=256)
    cls = ir.class_index[query.cls]
    e.set_option("prune", prune)
    st = e.sweep(cls, 5, 1)
    out[prune] = (e.download_assignment(cls, 0, 6000), e.download_assignment(cls, 52, 6000), e.download_logweights(cls, 6000), st)
    print(prune, st)
d0 = np.nonzero(out[1][0] != out[0][0])[0]; d1 = np.nonzero(out[1][1] != out[0][1])[0]
print('diff hosp rows', len(d0), d0[:20], 'diff measure rows', len(d1), d1[:20])
print('logw maxdiff', np.abs(out[1][2]-out[0][2]).max())
rows = list(d0[:4]) + list(d1[:4])
import ctypes as C
for prune in (1, 0):
    model, query, ir, dirty, truth, o, e = _setup_synth(cfg, n_rows=6000, H=256)
    cls = ir.class_index[query.cls]
    e.set_option("prune", prune)
    for r in rows:
        try:
            ke, we, se, me = e.row_move_debug(cls, int(r), 5, 1, 2)
            print('prune', prune, 'row', r, 'sel', se, 'ml', me, 'keys', ke[:8].tolist(), 'w', we[:3])
        except Exception as ex:
            print('prune', prune, 'row', r, 'ERR', ex)
        K, nv = 20, 67
        ch = (C.c_int32 * K)(); sc = (C.c_int32 * (K * nv))()
        e.L.pclean_debug_particles(e.h, int(r), 0, ch, sc)
        print('   choices', list(ch))
        for k in range(K):
            if ch[k] <= -2 and ch[k] != -3:
                row = sc[k*nv:(k+1)*nv]
                print('   particle', k, 'scratch', [(v+1, x) for v, x in enumerate(row) if x != -3][:45])
                print('      state cell (vertex 8):', row[7], repr(ir.strings[row[7]]) if 0 <= row[7] < len(ir.strings) else None)
                break
