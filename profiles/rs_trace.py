import os, sys, ctypes, numpy as np, torch
sys.path.insert(0, os.getcwd())
import bench
from autodriver_pointcloud_preprocessor_b200 import _capi, engine
msgs = bench.make_frames(2, seed0=0)
ctx = engine.Context(max_points=bench.N_POINTS)
fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=_capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True, transforms=[bench.TF], crop=bench.CROP)
pcfg = engine.make_pipeline_cfg(fcfg, **bench.STAGES)
for f in range(4):
    m = msgs[f % 2]
    data = torch.frombuffer(bytearray(m.data), dtype=torch.uint8).cuda()
    desc = engine.make_cloud_desc(m.fields, m.point_step, m.width, data)
    out, counts, plane = ctx.pipeline_run([desc], pcfg)
    ctx.check()
buf = (ctypes.c_uint64 * 8192)()
lib = ctypes.CDLL(_capi.LIB_PATH)
print("rc", lib.apc_debug_rs_trace(buf))
a = np.frombuffer(buf, dtype=np.uint64).reshape(1024, 8).astype(np.int64)
a = a[a[:, 0] > 0]
t0 = a[:, 0].min()
print("ctas", len(a))
d = a[:, :6] - t0
np.set_printoptions(linewidth=200)
print("start  min/med/max", d[:,0].min(), np.median(d[:,0]), d[:,0].max())
for k, name in [(1,"prologue"),(2,"scoring"),(3,"flush"),(4,"atom+ticket")]:
    x = a[:,k]-a[:,k-1]
    print(name, "min/med/max ns", x.min(), np.median(x), x.max())
print("end (stamp4) min/med/max", d[:,4].min(), np.median(d[:,4]), d[:,4].max())
col = a[a[:,5]>0]      # the last CTA of each chunk column: its column's tally sum
print("column sum ns", (col[:,5]-col[:,4]), "end at", col[:,5]-t0)
last = a[a[:,6]>0]     # the CTA of the last column: the selection
print("selection ns", (last[:,6]-last[:,5]), "end at", last[:,6]-t0)
buf2 = None
sm = a[:, 7]
order = np.argsort(sm, kind="stable")
print("sm  cta  start prologue scoring flush ticket(end)")
for i in order[:0]:
    print(int(sm[i]), int(i), d[i, :5].tolist())
