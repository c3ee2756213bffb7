"""Grid generation time on C2 with the host-side topology replay run synchronously and on its worker thread."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch as pt
import synth
import sparsespatialsampling_b200 as s3
from sparsespatialsampling_b200.s_cube import SamplingTree
n = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
x = synth.cylinder2d_cloud(n, seed=0)
m = synth.wake_metric(x.cuda()).cpu()
geoms = lambda: [s3.geometry.CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
                 s3.geometry.SphereGeometry("cylinder", False, synth.CYL2D["pos"], synth.CYL2D["radius"], refine=True)]
print("cpus", os.cpu_count(), "affinity", len(os.sched_getaffinity(0)))
for rep in range(3):
    for label, asyn in (("replay sync", False), ("replay async", True)):
        SamplingTree.topology_async = asyn
        tree = SamplingTree(x, m, geoms(), uniform_level=5, min_metric=0.75)
        pt.cuda.synchronize(); t0 = time.perf_counter(); tree.refine(); pt.cuda.synchronize(); t1 = time.perf_counter()
        i = tree.data_final_mesh
        print(f"rep {rep} {label:13s} total {t1-t0:.3f}s adaptive {i['t_adaptive']:.3f} renumber {i['t_renumbering']:.3f} cells {i['n_cells']}")
