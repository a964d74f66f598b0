"""The GPU parity tests, run on the CPU against a g++ build of the PRODUCT sources (tests/host_emu/build.py build_full: every
.cu of cup2d_b200/csrc with kernel launches turned into one OS thread per CUDA thread — real barriers, warp shuffles, shared
memory, atomics —, CUDA runtime calls mapped to malloc/memcpy and the handful of PTX statements (mbarrier / bulk copy /
reciprocal seed / system-scope loads and stores) replaced by their host meaning).

This checks the LOGIC of the kernels and of the host driver without a GPU — indexing, tables, reductions, the Krylov control
flow — not their execution on hardware (no launch configuration, no real asynchrony, no performance).  It is test
infrastructure: built on demand under tests/, never shipped, and not a CPU fallback of the product (cup2d_b200 still refuses to
run without its CUDA library; the emulated library is only ever loaded through the explicit CUP2D_B200_LIB override below).

A fast subset runs here; the whole suite: tools/run_emulated_gpu_tests.sh (about 5 minutes)."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

SUBSET = ("(operators_vs_reference_golden or uniformly_advected or vorticity_tagging or adapt_tags or dump_files or penalisation_phase or shape_calls "
          "or steps_L2_random_k8 or rectangular_domain or host_pipeline or degenerate or amr_bodies or amr_adapt_tags or amr_dump or (uniform_mesh_equals and True) or synthetic_three_level or amr_fast or amr_advect_diffuse or amr_pressure_gradient) "
          "and not reference_driver")


@pytest.fixture(scope="module")
def emulated_library():
    sys.path.insert(0, os.path.join(HERE, "host_emu"))
    import build
    return build.build_full()


def test_gpu_parity_subset_on_the_emulated_library(emulated_library):
    env = dict(os.environ, CUP2D_B200_LIB=emulated_library)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(HERE, "test_gpu_parity.py"),
                        os.path.join(HERE, "test_gpu_amr.py"), "-m", "gpu", "-q", "-x", "-k", SUBSET, "-p", "no:cacheprovider"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env, timeout=900, cwd=ROOT)
    tail = r.stdout[-1500:]
    assert r.returncode == 0, tail
    assert " passed" in tail and "failed" not in tail
    n = int(tail.split(" passed")[0].split()[-1])
    assert n >= 12, tail


def test_two_ranks_emulated_in_one_process(emulated_library):
    """the multi-GPU path (peer-memory halo pulls with ready flags, in-kernel all-reduce of the Krylov dots, SFC-range
    partition) with the two ranks running as threads of one process: their 'device' buffers are mapped into each other through
    the emulated IPC handles and their kernels really run concurrently.  2 steps x 10 Poisson iterations vs the oracle."""
    code = r'''
import sys, threading, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import cup2d_b200, cup2d_oracle as orc
W, L = 2, 3
N = 8 << L
x = (np.arange(N) + 0.5) / N
X, Y = np.meshgrid(x, x)
rng = np.random.default_rng(5)
u = np.sin(2 * np.pi * X) * np.cos(2 * np.pi * Y) + 0.05 * rng.uniform(-1, 1, (N, N))
v = -np.cos(2 * np.pi * X) * np.sin(2 * np.pi * Y) + 0.05 * rng.uniform(-1, 1, (N, N))
p = np.cos(2 * np.pi * X) * np.cos(2 * np.pi * Y)
bar, slots, res, errs = threading.Barrier(W), [None] * W, [None] * W, []
class Dist:                       # in-process stand-in for torch.distributed (only carries the opaque blobs)
    def __init__(self, rank): self.rank = rank
    def all_gather_object(self, out, obj):
        slots[self.rank] = obj; bar.wait()
        out[:] = slots; bar.wait()
    def barrier(self): bar.wait()
def run(rank):
    try:
        sim = cup2d_b200.Simulation(L, nu=1e-3, cfl=0.5, rank=rank, nranks=W)
        sim.attach_peers(Dist(rank))
        sim.upload("vel", u, v); sim.upload("pres", p)
        outs = []
        for s in range(2):
            dt, it, err = sim.step(max_iter=10)
            outs.append((dt, sim.download_blocks("vel"), sim.download_blocks("pres")))
            bar.wait()
        res[rank] = (sim.order, sim.nbx, sim.nby, outs)
        bar.wait(); sim.close()
    except Exception as e:
        errs.append(repr(e)); bar.abort()
ths = [threading.Thread(target=run, args=(r,)) for r in range(W)]
[t.start() for t in ths]; [t.join() for t in ths]
assert not errs, errs
order, nbx, nby, _ = res[0]
ru, rv, rp, worst = u, v, p, 0.0
for s in range(2):
    ref = orc.step(ru, rv, rp, 1e-3, 0.5, kiter=10)
    vel = np.concatenate([res[r][3][s][1] for r in range(W)]); pr = np.concatenate([res[r][3][s][2] for r in range(W)])
    gu, gv = cup2d_b200.from_blocks(vel, order, nbx, nby, 2); gp = cup2d_b200.from_blocks(pr, order, nbx, nby, 1)
    worst = max(worst, abs(res[0][3][s][0] - ref["dt"]) / ref["dt"], np.abs(gu - ref["u"]).max(), np.abs(gv - ref["v"]).max(),
                np.abs(gp - ref["p"]).max())
    ru, rv, rp = ref["u"], ref["v"], ref["p"]
print("WORST", worst)
assert worst < 1e-12
''' % (ROOT, os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900,
                       env=dict(os.environ, CUP2D_B200_LIB=emulated_library))
    assert r.returncode == 0 and "WORST" in r.stdout, r.stdout[-1500:]


def test_a_rank_that_never_arrives_fails_the_call_instead_of_hanging(emulated_library):
    """bounded cross-GPU waits: rank 1 attaches but never issues its step; rank 0's first halo wait runs into the time limit
    (CUP2D_COMM_TIMEOUT_MS), every later wait is skipped, and the call that synchronises reports CUP2D_ECOMM — the reference
    aborts through MPI in that situation, an unbounded spin would hang the GPU"""
    code = r'''
import sys, threading, time, numpy as np
sys.path.insert(0, %r)
import cup2d_b200
from cup2d_b200.lib import Cup2dError
W, L = 2, 3
N = 8 << L
u = np.random.default_rng(1).uniform(-1, 1, (N, N))
bar, slots, msg = threading.Barrier(W), [None] * W, []
class Dist:
    def __init__(self, rank): self.rank = rank
    def all_gather_object(self, out, obj):
        slots[self.rank] = obj; bar.wait()
        out[:] = slots; bar.wait()
    def barrier(self): bar.wait()
def run(rank):
    sim = cup2d_b200.Simulation(L, rank=rank, nranks=W)
    sim.attach_peers(Dist(rank))
    sim.upload("vel", u, u); sim.upload("pres", u)
    if rank == 0:
        t0 = time.time()
        try:
            sim.step(max_iter=4)
            msg.append("no error")
        except Cup2dError as e:
            msg.append(str(e)); msg.append(time.time() - t0)
    bar.wait()
ths = [threading.Thread(target=run, args=(r,)) for r in range(W)]
[t.start() for t in ths]; [t.join() for t in ths]
print("MSG", msg)
assert "timed out" in msg[0] and "-5" in msg[0] and msg[1] < 60
''' % (ROOT,)
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600,
                       env=dict(os.environ, CUP2D_B200_LIB=emulated_library, CUP2D_COMM_TIMEOUT_MS="300"))
    assert r.returncode == 0 and "MSG" in r.stdout, r.stdout[-1500:]


@pytest.mark.skipif(os.environ.get("CUP2D_TEST_SLOW") != "1",
                    reason="35 s; test_multi_level_steps_on_three_ranks_emulated runs the same constructor inside whole time steps")
def test_amr_poisson_matrix_distributed_over_three_ranks_emulated(emulated_library):
    """cup2d_poisson_create_general_ranks: the Poisson matrix of the reference's 7-level run.sh mesh (neighbour table +
    coarse-fine rows from the library's plan) distributed over three ranks by block ranges, the ranks running as threads of one
    process: remote blocks named by either table become halo slots refreshed by peer pulls, the Krylov kernels are the
    uniform path's.  8 iterations against the same solve on one rank."""
    code = r'''
import sys, threading, numpy as np
sys.path.insert(0, %r)
from cup2d_b200.amr import AmrPlan, DistributedPoisson
d = np.load(%r)
blocks = np.ascontiguousarray(d["blocks"], dtype=np.int32)
nb = len(blocks)
nbr, rows, rowptr, col, val = AmrPlan(blocks, int(d["bpdx"]), int(d["bpdy"])).poisson()
rng = np.random.default_rng(7)
b, x0 = rng.uniform(-1, 1, (nb, 64)), rng.uniform(-0.1, 0.1, (nb, 64))
one = DistributedPoisson(nbr, rows, rowptr, col, val, [0, nb], 0); one.attach_peers()
xs, its, errs_ = one.solve(b, x0, max_iter=8); one.close()
W, rb = 3, [0, 90, 190, nb]
bar, slots, res, errs = threading.Barrier(W), [None] * W, [None] * W, []
class Dist:
    def __init__(self, rank): self.rank = rank
    def all_gather_object(self, out, obj):
        slots[self.rank] = obj; bar.wait(); out[:] = slots; bar.wait()
    def barrier(self): bar.wait()
def run(rank):
    try:
        p = DistributedPoisson(nbr, rows, rowptr, col, val, rb, rank)
        p.attach_peers(Dist(rank))
        res[rank] = p.solve(b[rb[rank]:rb[rank + 1]], x0[rb[rank]:rb[rank + 1]], max_iter=8)
        bar.wait(); p.close()
    except Exception as e:
        errs.append(repr(e)); bar.abort()
ths = [threading.Thread(target=run, args=(r,)) for r in range(W)]
[t.start() for t in ths]; [t.join() for t in ths]
assert not errs, errs
x = np.concatenate([r[0] for r in res])
worst = np.abs(x - xs).max() / np.abs(xs).max()
print("WORST", worst, [r[1] for r in res], its)
assert worst < 1e-10 and all(r[1] == 8 for r in res) and its == 8 and abs(res[0][2] - errs_) < 1e-10
''' % (ROOT, os.path.join(ROOT, "tests", "golden", "amrlab_lmax8.npz"))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900,
                       env=dict(os.environ, CUP2D_B200_LIB=emulated_library))
    assert r.returncode == 0 and "WORST" in r.stdout, r.stdout[-1500:]


@pytest.mark.skipif(os.environ.get("CUP2D_TEST_SLOW") != "1", reason="first (replicated-operators) form; the distributed form below is the default test")
def test_multi_level_steps_on_three_ranks_emulated(emulated_library):
    """several GPUs on a multi-level mesh, first form (cup2d_amr_set_ranks): every rank holds the whole mesh and computes the
    stencil operators redundantly, the Poisson solve is distributed by block ranges and all-gathered through the peers' arrays.
    Three ranks (uneven block ranges) as threads of one process, 2 steps x 5 iterations on a three-level mesh: all ranks
    bitwise identical, and equal to the one-rank run to rounding."""
    code = r'''
import sys, threading, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench_amr
from cup2d_b200.amr import AmrSimulation
blocks = bench_amr.three_level_mesh(3, r1=0.3, r2=0.15, centre=(0.45, 0.55))
nb, h0, nu = len(blocks), 1 / 8, 1e-3
rng = np.random.default_rng(3)
vel, pres = bench_amr.seeded_fields(blocks, h0)
vel, pres = vel + 0.05 * rng.uniform(-1, 1, vel.shape), pres + 0.05 * rng.uniform(-1, 1, pres.shape)
def steps(sim):
    out = []
    sim.set_fast(True); sim.upload("vel", vel); sim.upload("pres", pres)
    for s in range(2):
        info = sim.step(cfl=0.5, max_iter=5)
        out.append((info, sim.download("vel"), sim.download("pres")))
    return out
one = AmrSimulation(blocks, 1, 1, h0, nu); ref = steps(one); one.close()
W = 3
rb = [0, nb // 3 + 7, 2 * nb // 3 - 5, nb]
bar, slots, res, errs = threading.Barrier(W), [None] * W, [None] * W, []
class Dist:
    def __init__(self, rank): self.rank = rank
    def all_gather_object(self, out, obj):
        slots[self.rank] = obj; bar.wait(); out[:] = slots; bar.wait()
    def barrier(self): bar.wait()
def run(rank):
    try:
        sim = AmrSimulation(blocks, 1, 1, h0, nu)
        sim.set_ranks(rank, rb, Dist(rank))
        res[rank] = steps(sim)
        bar.wait(); sim.close()
    except Exception as e:
        errs.append(repr(e)); bar.abort()
ths = [threading.Thread(target=run, args=(r,)) for r in range(W)]
[t.start() for t in ths]; [t.join() for t in ths]
assert not errs, errs
worst = 0.0
for s in range(2):
    assert all(np.array_equal(res[0][s][1], res[r][s][1]) and np.array_equal(res[0][s][2], res[r][s][2]) and res[0][s][0] == res[r][s][0] for r in range(W))
    worst = max(worst, np.abs(res[0][s][1] - ref[s][1]).max() / np.abs(ref[s][1]).max(),
                np.abs(res[0][s][2] - ref[s][2]).max() / np.abs(ref[s][2]).max(), abs(res[0][s][0][0] - ref[s][0][0]))
print("WORST", worst)
assert worst < 1e-11
''' % (ROOT, os.path.join(ROOT, "tools"))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900,
                       env=dict(os.environ, CUP2D_B200_LIB=emulated_library))
    assert r.returncode == 0 and "WORST" in r.stdout, r.stdout[-1500:]


def test_distributed_multi_level_mesh_on_three_ranks_emulated(emulated_library):
    """several GPUs on a multi-level mesh, second form (cup2d_amr_create_ranks): the mesh itself is distributed by block ranges;
    every rank holds its blocks plus halo slots for the remote blocks its tables name (face neighbours, ghost-row sources, fine
    sides of its coarse faces, Poisson columns), refreshed by whole-block peer pulls; face fluxes cross rank boundaries inside a
    field array; dt and the pressure means are all-reduced in a kernel.  Three ranks (uneven ranges) as threads of one process:
    (1) on the reference's 7-level run.sh mesh the body sums / blend / u_def assembly against the one-rank context and the
    flux-corrected operators and adapt()'s tagging field against the reference's own outputs; (2) two full steps on a
    three-level mesh against the one-rank run."""
    code = r'''
import sys, threading, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench_amr
from cup2d_b200.amr import AmrSimulation
W = 3
bar, slots, errs = threading.Barrier(W), [None] * W, []
class Dist:
    def __init__(self, rank): self.rank = rank
    def all_gather_object(self, out, obj):
        slots[self.rank] = obj; bar.wait(); out[:] = slots; bar.wait()
    def barrier(self): bar.wait()
def on_ranks(fn):
    res = [None] * W
    def run(rank):
        try:
            res[rank] = fn(rank); bar.wait()
        except Exception as e:
            errs.append(repr(e)); bar.abort()
    ths = [threading.Thread(target=run, args=(r,)) for r in range(W)]
    [t.start() for t in ths]; [t.join() for t in ths]
    assert not errs, errs
    return res
# (1) operators on the reference's mesh
d = dict(np.load(%r))   # read everything now: the lazy NpzFile is not safe to read from several threads
blocks = np.ascontiguousarray(d["blocks"], dtype=np.int32); nb = len(blocks); rb = [0, 81, 199, nb]
rng = np.random.default_rng(11)
ids = np.sort(rng.choice(nb, 40, replace=False)).astype(np.int32)      # a body whose obstacle blocks lie on all three ranks
X, ud = rng.uniform(-0.3, 1.0, (len(ids), 8, 8)), rng.uniform(-1, 1, (len(ids), 8, 8, 2))
body = (1e7, float(d["dt"]), 0.9, 0.5)
one = AmrSimulation(blocks, int(d["bpdx"]), int(d["bpdy"]), float(d["h0"]), float(d["nu"]))
one.upload("vel", d["vel"]); one.upload("chi", d["chi"]); one.shape_set(0, ids, X, ud)
want_q = one.shape_integrals(0, *body)
one.penalize(0, *body, 0.1, -0.2, 0.7); want_v = one.download("vel"); one.udef_assemble(); want_t = one.download("tmpV")
one.close()
def ops(rank):
    sl, dt = slice(rb[rank], rb[rank + 1]), float(d["dt"])
    sim = AmrSimulation.distributed(blocks, int(d["bpdx"]), int(d["bpdy"]), float(d["h0"]), float(d["nu"]), rank, rb, Dist(rank))
    mine = (ids >= rb[rank]) & (ids < rb[rank + 1])
    sim.upload("vel", d["vel"][sl]); sim.upload("chi", d["chi"][sl]); sim.shape_set(0, ids[mine] - rb[rank], X[mine], ud[mine])
    q = sim.shape_integrals(0, *body)                                   # all-reduced: the same seven sums on every rank
    sim.penalize(0, *body, 0.1, -0.2, 0.7); pv = sim.download("vel"); sim.udef_assemble(); pt = sim.download("tmpV")
    assert np.abs(q - want_q).max() <= 1e-12 * np.abs(want_q).max() and np.array_equal(pv, want_v[sl]) and np.array_equal(pt, want_t[sl])
    sim.upload("vel", d["vel"][sl]); sim.advect_diffuse_rhs(dt); adv = sim.download("tmpV")
    sim.upload("tmpV", d["udef"][sl]); sim.upload("chi", d["chi"][sl]); sim.upload("pold", d["pres"][sl])
    sim.pressure_rhs(dt, True); rhs1 = sim.download("tmp")
    sim.upload("pres", d["pres"][sl]); sim.pressure_gradient(dt); gp = sim.download("tmpV")
    bar.wait(); sim.close()
    return adv, rhs1, gp
res = on_ranks(ops)
worst = 0.0
for i, name in enumerate(("adv", "rhs1", "gradp")):
    got = np.concatenate([res[r][i] for r in range(W)])
    worst = max(worst, np.abs(got - d[name]).max() / np.abs(d[name]).max())
# (1b) adapt()'s tagging field on the reference's mesh with its fish
g = dict(np.load(%r))
def tags(rank):
    sl = slice(rb[rank], rb[rank + 1])
    sim = AmrSimulation.distributed(blocks, int(g["bpdx"]), int(g["bpdy"]), float(g["h0"]), 4e-5, rank, rb, Dist(rank))
    sim.upload("vel", g["vel"][sl]); sim.upload("chi", g["chi"][sl])
    out = (sim.adapt_tags(float(g["rtol"]), int(g["level_max"])), sim.download("tmp"))
    bar.wait(); sim.close()
    return out
assert np.array_equal(g["blocks"], d["blocks"])
res = on_ranks(tags)
field = np.concatenate([res[r][1] for r in range(W)]).reshape(nb, 8, 8); linf = np.concatenate([res[r][0] for r in range(W)])
wl = np.abs(g["tagfield"]).reshape(nb, -1).max(axis=1)
worst = max(worst, np.abs(field - g["tagfield"]).max() / np.abs(g["tagfield"]).max())
assert np.array_equal(linf > g["rtol"], wl > g["rtol"]) and np.array_equal(linf < g["ctol"], wl < g["ctol"])
# (2) full steps
mb = bench_amr.three_level_mesh(3, r1=0.3, r2=0.15, centre=(0.45, 0.55)); mn = len(mb); h0 = 1 / 8
rng = np.random.default_rng(3)
vel, pres = bench_amr.seeded_fields(mb, h0)
vel, pres = vel + 0.05 * rng.uniform(-1, 1, vel.shape), pres + 0.05 * rng.uniform(-1, 1, pres.shape)
def steps(sim, sl):
    out = []
    sim.upload("vel", vel[sl]); sim.upload("pres", pres[sl])
    for s in range(2):
        info = sim.step(cfl=0.5, max_iter=5)
        out.append((info, sim.download("vel"), sim.download("pres")))
    return out
one = AmrSimulation(mb, 1, 1, h0, 1e-3); one.set_fast(True); ref = steps(one, slice(0, mn)); one.close()
mrb = [0, mn // 3 + 7, 2 * mn // 3 - 5, mn]
def dsteps(rank):
    sim = AmrSimulation.distributed(mb, 1, 1, h0, 1e-3, rank, mrb, Dist(rank))
    out = steps(sim, slice(mrb[rank], mrb[rank + 1]))
    bar.wait(); sim.close()
    return out
res = on_ranks(dsteps)
for s in range(2):
    v = np.concatenate([res[r][s][1] for r in range(W)]); p = np.concatenate([res[r][s][2] for r in range(W)])
    worst = max(worst, np.abs(v - ref[s][1]).max() / np.abs(ref[s][1]).max(), np.abs(p - ref[s][2]).max() / np.abs(ref[s][2]).max(),
                abs(res[0][s][0][0] - ref[s][0][0]) / ref[s][0][0])
    assert all(res[r][s][0] == res[0][s][0] for r in range(W)) and res[0][s][0][1] == ref[s][0][1] == 5
print("WORST", worst)
assert worst < 1e-11
''' % (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests", "golden", "amrlab_lmax8.npz"),
       os.path.join(ROOT, "tests", "golden", "amrtags_lmax8.npz"))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300,  # a rank that dies leaves the others spinning on its flags
                      
                       env=dict(os.environ, CUP2D_B200_LIB=emulated_library))
    assert r.returncode == 0 and "WORST" in r.stdout, r.stdout[-1500:]


# The two sanitizer builds recompile every product source with -fsanitize and take 4-6 minutes on 8 cores: they run when asked
# for (CUP2D_TEST_SANITIZERS=1, as tools/run_emulated_gpu_tests.sh does); the hardware counterpart is compute-sanitizer
# memcheck/racecheck on the GPU box (profiles/r02a_sanitizer_*).
sanitizers = pytest.mark.skipif(os.environ.get("CUP2D_TEST_SANITIZERS") != "1", reason="sanitizer builds are opt-in: CUP2D_TEST_SANITIZERS=1")


@sanitizers
def test_no_data_races_under_thread_sanitizer():
    """race hunt: the emulated product sources rebuilt with -fsanitize=thread run a uniform-grid time step (advect with its
    staged loads, pressure kernels, the Krylov kernels with their grid reductions, the chi-mask tags) and the multi-level step
    on baseline and fast kernels.  Every CUDA thread being an OS thread, an access pair not ordered by a barrier, shuffle or
    atomic is a ThreadSanitizer report (checked by hand: removing the __syncwarp between the two passes of the multi-level
    advect kernel produces reports at its partial-result planes).  None is expected."""
    sys.path.insert(0, os.path.join(HERE, "host_emu"))
    import build
    try:
        exe = build.build_tsan()
    except subprocess.CalledProcessError:
        pytest.skip("ThreadSanitizer runtime not available to g++ on this box")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800,
                       env=dict(os.environ, TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0"))
    assert r.returncode == 0, r.stdout[-3000:]
    assert "ThreadSanitizer" not in r.stdout, r.stdout[-3000:]
    assert r.stdout.count("multi-level step") == 2 and "uniform step" in r.stdout and "bodies / tags / dump" in r.stdout


@sanitizers
def test_no_out_of_bounds_or_misaligned_access_under_address_sanitizer(golden_dir, tmp_path):
    """memcheck stand-in: the same driver built with -fsanitize=address,alignment,bounds.  Every emulated device buffer and
    every __shared__ array is its own exact-size allocation filled with 0xFF bytes (cudaMalloc does not zero), the vector
    types carry the alignment their hardware loads need (double2 / int4 / float4: 16 bytes) and cp.async.bulk checks its
    16-byte rule: an overrun, a misaligned vector access or a NaN from never-written memory ends the run.  Uniform step +
    multi-level step (baseline, fast) on the small two-level mesh; with CUP2D_TEST_SLOW=1 also on the reference's 278-block
    7-level run.sh mesh (7 minutes; clean when this was written)."""
    import numpy as np
    sys.path.insert(0, os.path.join(HERE, "host_emu"))
    import build
    try:
        exe = build.build_tsan(sanitize="address,alignment,bounds")
    except subprocess.CalledProcessError:
        pytest.skip("AddressSanitizer runtime not available to g++ on this box")
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800, env=env)
    assert r.returncode == 0 and "runtime error" not in r.stdout and "AddressSanitizer" not in r.stdout, r.stdout[-3000:]
    assert r.stdout.count("multi-level step") == 2 and "uniform step" in r.stdout and "nan" not in r.stdout.lower()
    assert "bodies / tags / dump" in r.stdout
    if os.environ.get("CUP2D_TEST_SLOW") == "1":
        d = np.load(os.path.join(golden_dir, "amrlab_lmax8.npz"))
        mesh = tmp_path / "mesh.bin"
        np.ascontiguousarray(d["blocks"], dtype=np.int32).tofile(mesh)
        r = subprocess.run([exe, str(mesh), str(int(d["bpdx"])), str(int(d["bpdy"])), repr(float(d["h0"]))], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=3000, env=env)
        assert r.returncode == 0 and r.stdout.count("mesh step") == 2, r.stdout[-3000:]


def test_measurement_variants_keep_parity():
    """the build switches of the advect stage that are OFF in the default build (advect.cu: CUP2D_ADV_LDGSTS=0 — the tile
    filled by per-row bulk copies on one mbarrier instead of cp.async; CUP2D_ADV_SPECIALIZE=0 — one copy of the line code with
    run-time strides for both passes; CUP2D_ADV_FASTPATH=0 — every line through the general core) built together into an
    emulated library: the operator / advect / time-step parity tests still pass.  (Each was also run on hardware:
    profiles/r02e_variants.jsonl, r02g_variants.jsonl.)"""
    sys.path.insert(0, os.path.join(HERE, "host_emu"))
    import build
    lib = build.build_full(("CUP2D_ADV_LDGSTS=0", "CUP2D_ADV_SPECIALIZE=0", "CUP2D_ADV_FASTPATH=0"), "_variants")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(HERE, "test_gpu_parity.py"), "-m", "gpu", "-q", "-x", "-k",
                        "(operators_vs_reference_golden or steps_L2_random_k8 or rectangular_domain or advect_stage_vs_oracle or uniformly_advected) "
                        "and not reference_driver", "-p", "no:cacheprovider"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=dict(os.environ, CUP2D_B200_LIB=lib),
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout[-1500:]


def _emulated_driver(name, emulated_library, tmp_path):
    """oracle/_ref/<name>.o (the reference's loop with the drop-in fragments spliced in, compiled by build()) linked against the
    emulated library.  Only the link step runs here, so the reference's sources are not needed, only what build() left in
    oracle/_ref/; skipped where that was not built."""
    objs = [os.path.join(ROOT, "oracle", "_ref", f) for f in (name + ".o", "ref_spmat_cpu.o")]
    if not all(os.path.exists(o) for o in objs):
        pytest.skip(f"oracle/_ref/{name}.o not built")
    emu_dir = os.path.dirname(emulated_library)
    exe = str(tmp_path / (name + "_emu"))
    subprocess.run(["g++", "-fopenmp", "-o", exe, *objs, f"-L{emu_dir}", "-lcup2d_emu", f"-Wl,-rpath,{emu_dir}"], check=True)
    return exe


def _reference_harness():
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_harness not built")
    return exe


@pytest.mark.parametrize("name", ["steps_L2_random_k8", "steps_L3_tg_k15"])
def test_reference_time_loop_on_the_emulated_library(emulated_library, golden_dir, name, tmp_path):
    """the drop-in boundary for the operators, end to end: the reference's OWN time loop (unmodified main.cpp with lines
    6607-6642 and 7007-7187 replaced at build time by dropin/patched_loop_*.inc + dropin/b200_loop_glue.h), linked against the
    emulated library, against the steps the unmodified reference produced (tests/golden/steps_*.npz)"""
    import numpy as np
    exe = _emulated_driver("ref_harness_patched", emulated_library, tmp_path)
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    L, K, ns = int(g["L"]), int(g["kiter"]), len(g["dt"])
    N = 8 << L
    z = np.zeros((N, N))
    fin, fout = tmp_path / "in.bin", tmp_path / "out.bin"
    np.concatenate([a.ravel() for a in (g["u0"], g["v0"], g["p0"], z, z, z)]).tofile(fin)
    subprocess.run([exe, "steps", str(L), repr(float(g["nu"])),
                    repr(float(g["cfl"])), str(ns), str(K), str(fin), str(fout)], check=True, stderr=subprocess.DEVNULL,
                   env=dict(os.environ, OMP_NUM_THREADS="1", CUP2D_B200_MAX_ITER=str(K)), timeout=900)
    raw = np.fromfile(fout).reshape(ns, 1 + 5 * N * N)
    f = raw[:, 1:].reshape(ns, 5, N, N)
    assert np.abs(raw[:, 0] - g["dt"]).max() < 1e-15
    assert np.abs(f[:, 0] - g["u"]).max() < 1e-12 and np.abs(f[:, 1] - g["v"]).max() < 1e-12
    assert np.abs(f[:, 2] - g["p"]).max() < 1e-10


def test_reference_loop_with_bodies_device_resident_on_the_emulated_library(emulated_library, tmp_path):
    """the device-resident form of the drop-in, WITH bodies: the reference's own loop with RK2, the penalisation sums, the
    blend, the u_def assembly and the pressure section on the library (dropin/resident_*.inc over main.cpp:6607-6642, 6648-6679,
    6945-6979, 6981-7187) while ongrid(), the 3x3 rigid-motion solve, the collision model and the forces stay on the host —
    two interacting fish, 4 steps (the last one with a collision), against the unmodified reference run the same way"""
    import numpy as np
    exes = (_reference_harness(), _emulated_driver("ref_harness_resident", emulated_library, tmp_path))
    env = dict(os.environ, OMP_NUM_THREADS="1", CUP2D_B200_MAX_ITER="5",
               CUP2D_REF_SHAPES="angle=0 L=0.8 xpos=0.52 ypos=0.44\n angle=175 L=0.8 xpos=0.47 ypos=0.56")
    outs = []
    for exe in exes:
        out = tmp_path / (os.path.basename(exe) + ".bin")
        subprocess.run([exe, "fsteps", "4", "4", "5", str(out)], check=True,
                       stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL, env=env, timeout=900)
        outs.append(np.fromfile(out))
    N = 128
    a, b = (o.reshape(-1, 1 + 3 * N * N + 10) for o in outs)
    assert a.shape == b.shape and len(a) == 4
    assert np.abs(a[:, 0] - b[:, 0]).max() < 1e-15                      # dt
    assert np.abs(a[:, 1:-10] - b[:, 1:-10]).max() < 1e-12              # u, v, p
    assert np.abs(a[:, -10:] - b[:, -10:]).max() < 1e-12                # centre of mass, u, v, omega of both fish
    assert np.abs(a[-1, 1:1 + N * N]).max() > 0.1                       # the fish really drive the flow


def _parse_asteps(path):
    import numpy as np
    a, i, out = np.fromfile(path), 0, []
    while i < len(a):
        dt, nb = a[i], int(a[i + 1])
        i += 2
        mesh = a[i:i + 3 * nb].reshape(nb, 3).astype(int)
        i += 3 * nb
        vel, pres = a[i:i + 128 * nb], a[i + 128 * nb:i + 192 * nb]
        i += 192 * nb
        out.append((dt, mesh, vel, pres))
    return out


@pytest.mark.parametrize("form,steps", [("amrloop", 2), ("amrresident", 3)])
def test_reference_amr_case_on_the_multi_level_path_emulated(emulated_library, tmp_path, form, steps):
    """config C1 end to end: the reference's own run.sh case (two fish, 7 refinement levels, 278 blocks, its own adapt() /
    ongrid() on the host) on the multi-level path of the library (fast kernels, Poisson rows from the library's own plan),
    linked against the emulated library, against the unmodified reference: same mesh and fields to rounding at every step.
      amrloop      RK2 and the whole pressure section on cup2d_amr, penalisation on the host (dropin/amr_loop_*.inc)
      amrresident  additionally the penalisation sums, the blend and the u_def assembly on the device
                   (cup2d_amr_shape_*, dropin/amr_resident_*.inc): the velocity crosses PCIe once each way per step
    (By hand, both forms: 13 steps across a regrid 278 -> 281 blocks stay within 3e-15 / 1.3e-14 relative in velocity /
    pressure.)"""
    import numpy as np
    exes = (_reference_harness(), _emulated_driver(f"ref_harness_{form}", emulated_library, tmp_path))
    # amrresident also takes adapt()'s tagging field from the device (cup2d_amr_adapt_tags, eleven adapt() calls in this
    # short run, the initial refinement included): the mesh must be the reference's from the start
    env = dict(os.environ, OMP_NUM_THREADS="1", CUP2D_B200_MAX_ITER="5", CUP2D_B200_AMR_FAST="1", CUP2D_B200_AMR_TAGS="1")
    runs = []
    for exe in exes:
        out = tmp_path / (os.path.basename(exe) + ".bin")
        subprocess.run([exe, "asteps", "8", str(steps), "5", str(out)], check=True,
                       stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL, env=env, timeout=1500)
        runs.append(_parse_asteps(out))
    assert len(runs[0]) == len(runs[1]) == steps
    for (dt0, m0, v0, p0), (dt1, m1, v1, p1) in zip(*runs):
        assert m0.shape == m1.shape and (m0 == m1).all() and len(set(m0[:, 0].tolist())) >= 5
        assert abs(dt0 - dt1) < 1e-15
        assert np.abs(v0 - v1).max() < 1e-12 * np.abs(v0).max()
        assert np.abs(p0 - p1).max() < 1e-11 * max(np.abs(p0).max(), 1e-300)
