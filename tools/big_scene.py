"""Scratch: build time (host SAH vs device LBVH, PLOC and binned SAH) and trace throughput on a large random scene."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import rttnw_b200 as R
from rttnw_b200 import abi, scene as S

n = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
rng = np.random.default_rng(5)
mat = S.Lambertian((0.5, 0.5, 0.5))
side = n ** (1 / 3) * 3.0
t0 = time.perf_counter()
items = [S.Sphere(tuple(c), float(r), mat) for c, r in zip(rng.uniform(-side, side, (n, 3)), rng.uniform(0.2, 1.0, n))]
desc = S.Scene(S.List(items)).to_desc()
print(f"{n} spheres: description built in {time.perf_counter() - t0:.2f} s", flush=True)
ctx = R.Context(0)
m = 2_000_000
o = rng.uniform(-side, side, (m, 3)); tgt = rng.uniform(-side, side, (m, 3))
rays = np.zeros(m, dtype=abi.RAY_DTYPE)
rays["origin"], rays["direction"] = o, tgt - o
rays["t_min"], rays["t_max"], rays["xi"] = 0.001, np.finfo(np.float64).max, 0.5
d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
d_hits = torch.empty(m * 88, dtype=torch.uint8, device="cuda")
res = {}
device = ("lbvh", "ploc", "sah_device")
kinds = ((("sah",) if n <= 1_000_000 else ()) + device) * 2
for kind in kinds:
    ctx.set_bvh_builder(kind)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    sc = R.DeviceScene(ctx, desc)
    torch.cuda.synchronize(); t1 = time.perf_counter()
    for _ in range(2): sc.trace_device(d_rays, d_hits, m)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); sc.trace_device(d_rays, d_hits, m); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    h = d_hits.cpu().numpy().view(abi.HIT_DTYPE)
    res[kind] = h.copy()
    st = sc.trace_stats(d_rays, m)
    print(f"{kind:10s}: scene create {1e3 * (t1 - t0):8.1f} ms ({sc.info()['bvh_nodes']} nodes), trace {m} rays {ms:.2f} ms = {m / ms / 1e6:.2f} Grays/s, hits {np.mean(h['prim_id'] >= 0):.3f}, "
          f"{st['node_visits']:.1f} node visits and {st['sphere_tests']:.2f} sphere tests per ray", flush=True)
    sc.close()
for k in res:
    if k != "lbvh": print(f"same primitive under {k} and lbvh trees: {(res[k]['prim_id'] == res['lbvh']['prim_id']).mean():.6f}")
