"""Every entry point once on small inputs -- meant to run under compute-sanitizer:
   compute-sanitizer --tool memcheck  python tools/sanitize_small.py
   compute-sanitizer --tool racecheck python tools/sanitize_small.py
   compute-sanitizer --tool initcheck python tools/sanitize_small.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import pcu_b200 as pcu

rng = np.random.default_rng(0)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 6000
x = rng.random((n, 3)).astype(np.float32)
y = rng.random((n + 137, 3)).astype(np.float32)
lat = np.stack(np.meshgrid(*[np.arange(12)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32) / 12   # ties everywhere


def step(name, fn):
    out = fn()
    torch.cuda.synchronize()
    print("ok", name, flush=True)
    return out


step("knn k=1", lambda: pcu.k_nearest_neighbors(x, y, 1))
step("knn k=16", lambda: pcu.k_nearest_neighbors(x, y, 16))
step("knn k=5 fp64", lambda: pcu.k_nearest_neighbors(x.astype(np.float64), y.astype(np.float64), 5))
step("knn k=40 (pyramid path)", lambda: pcu.k_nearest_neighbors(x[:2000], y, 40))
step("knn lattice k=8 (tie replay)", lambda: pcu.k_nearest_neighbors(lat + 0.01, lat, 8))
step("knn far apart", lambda: pcu.k_nearest_neighbors(x + 50.0, y, 4))
step("knn tiny clouds (one-CTA binning)", lambda: pcu.k_nearest_neighbors(x[:300], y[:200], 3))
step("chamfer", lambda: pcu.chamfer_distance(x, y))
step("chamfer return_index", lambda: pcu.chamfer_distance(x, y, return_index=True))
step("hausdorff", lambda: pcu.hausdorff_distance(x, y, return_index=True))
step("hausdorff lattice (witness replay)", lambda: pcu.hausdorff_distance(lat + 0.5 / 12, lat, return_index=True))
step("one-sided hausdorff fp64", lambda: pcu.one_sided_hausdorff_distance(x.astype(np.float64), y.astype(np.float64)))
xt, yt = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
step("device tensors chamfer", lambda: float(pcu.chamfer_distance(xt, yt)))
step("batched chamfer", lambda: pcu.batched_chamfer_distance(rng.random((6, 900, 3), dtype=np.float32), rng.random((6, 1100, 3), dtype=np.float32)))
step("batched chamfer (grid-wide binning)", lambda: pcu.batched_chamfer_distance(rng.random((2, 9000, 3), dtype=np.float32), rng.random((2, 9100, 3), dtype=np.float32)))
prep = step("prepare_cloud", lambda: pcu.prepare_cloud(y))
step("chamfer against a prepared cloud", lambda: pcu.chamfer_distance(x, prep))
step("hausdorff against a prepared cloud", lambda: pcu.one_sided_hausdorff_distance(x, prep))
v = rng.normal(size=(n, 3)); v /= np.linalg.norm(v, axis=1, keepdims=True)
step("normals knn", lambda: pcu.estimate_point_cloud_normals_knn(v.astype(np.float32), 10, v.astype(np.float32), np.deg2rad(30)))
step("normals ball", lambda: pcu.estimate_point_cloud_normals_ball(v.astype(np.float32), 0.01, v.astype(np.float32), np.deg2rad(30), 5, weight_function="rbf"))
step("normals ball, capped, fp64", lambda: pcu.estimate_point_cloud_normals_ball(v, 0.01, max_pts_per_ball=6))
step("voxel down-sampling", lambda: pcu.downsample_point_cloud_on_voxel_grid(0.05, x, x.astype(np.float64)))
step("poisson-disk down-sampling, radius and target", lambda: (pcu.downsample_point_cloud_poisson_disk(x, 0.05, random_seed=3),
                                                               pcu.downsample_point_cloud_poisson_disk(v, 0., target_num_samples=300, random_seed=3)))
step("deduplicate points", lambda: pcu.deduplicate_point_cloud(np.concatenate([x, x[:500]]), 1e-6))
step("deduplicate mesh fp64", lambda: pcu.deduplicate_mesh_vertices(np.concatenate([x, x[:500]]).astype(np.float64), rng.integers(0, n, (3000, 3)).astype(np.int64), 0.0))
pts_i = rng.integers(-1000, 1000, (n, 3)).astype(np.int32)
codes = step("morton encode", lambda: pcu.morton_encode(pts_i))
step("morton decode", lambda: pcu.morton_decode(codes))
step("morton add", lambda: pcu.morton_add(codes, codes))
step("morton knn", lambda: pcu.morton_knn(np.sort(codes), codes[:500], 7))
a = rng.random((40, 3)); b = rng.random((50, 3))
M = step("pairwise distances", lambda: pcu.pairwise_distances(a, b))
step("sinkhorn", lambda: pcu.sinkhorn(np.full(40, 1 / 40), np.full(50, 1 / 50), M, eps=1e-2, max_iters=50))
step("earth mover's distance", lambda: pcu.earth_movers_distance(a, b, eps=1e-2, max_iters=50))
print("done")
