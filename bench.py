#!/usr/bin/env python
"""bench.py -- Hψ applies/s (and SCF-step pieces) of the B200 plane-wave Kohn-Sham hot path.

Contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line
(rank 0).  A *step* is one full Hamiltonian application `mul!(Hψ, H::DftHamiltonianBlock, ψ)` on the block
of M bands of one k-block (batched FFT local part + kinetic + nonlocal P D P†ψ).

Workload at N=1: BASELINE.json configs[2] -- Si 5x5x5 supercell (250 atoms, 1000 e-), LDA, Γ only,
Ecut = 30 Ha, fft 192³, N_pw = 264 859, M = 503 bands, n_proj = 1250 (the configuration the north-star
targets are quoted on).  For N>1 every rank owns one k-block of that shape (k-points shard; weak scaling):
no data-path collective inside Hψ; the density allreduce of an SCF step is timed separately.

`value`  = band-applies/s with ψ/Hψ resident in HBM (CUDA events, max over ranks).
`e2e`    = the same call through the C ABI with pinned HOST ψ/Hψ buffers (H2D + D2H inside the timed region).
`roofline` = the Hψ-local kernel group (5 FFT-pipeline kernels per band chunk; HBM bound, algorithmic bytes
             72·N_fft + 40·N_pw per band, SURVEY §8d) against MEASURED_PEAKS.json hbm_gbs.
`roofline_gemm` = the nonlocal P D P†ψ GEMMs (FP64 DMMA; 16·N_pw·n_proj·M flop) against a cuBLAS ZGEMM
             probe measured in the same run (MEASURED_PEAKS.json has no FP64 figure).
`cpu_baseline` = the CPU oracle (port of the reference's band-at-a-time algorithm) on a bounded sample.

`--dump-outputs DIR` writes Hψ of the last timed step to DIR/hpsi.npy so that two builds can be compared output for output:
ψ and the operator depend only on the arguments (seeded generator), so the same arguments give the same inputs.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def effective_cpus():
    """CPUs usable by this process (affinity and cgroup quota aware; os.cpu_count() reports the whole host)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    return n


# BLAS / OpenMP pools sized to the CPUs we may really use (must happen before numpy / torch are imported)
_threads = max(1, effective_cpus() // max(1, int(os.environ.get("WORLD_SIZE", "1"))))
for _v in ("OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, str(_threads))
os.environ.setdefault("OMP_WAIT_POLICY", "passive")   # spinning OpenMP workers starve cuSOLVER's host stages (see dftk_b200/__init__.py)
if os.environ.get("OMP_NUM_THREADS") in (None, "1"):
    os.environ["OMP_NUM_THREADS"] = str(min(16, _threads))
import numpy as np

A_SI = 10.26 / 2
WORKLOADS = {
    # name: (supercell repeat, Ecut, n_bands)
    "si250": dict(rep=5, Ecut=30.0, desc="Si 5x5x5 supercell (250 atoms) LDA Gamma Ecut=30 Ha, fft 192^3"),
    "si16": dict(rep=2, Ecut=30.0, desc="Si 2x2x2 supercell (16 atoms) LDA Gamma Ecut=30 Ha (dev/smoke size)"),
    "si2": dict(rep=1, Ecut=30.0, desc="Si 2-atom primitive LDA Ecut=30 Ha (dev/smoke size)"),
}


def supercell(rep):
    lat = rep * np.array([[0, A_SI, A_SI], [A_SI, 0, A_SI], [A_SI, A_SI, 0]])
    pos = []
    for i in range(rep):
        for j in range(rep):
            for k in range(rep):
                for b in (np.ones(3) / 8, -np.ones(3) / 8):
                    pos.append((b + np.array([i, j, k])) / rep)
    return lat, pos


def n_bands_for(n_atoms):
    n_occ = 2 * n_atoms          # 4 e- per Si, doubly occupied
    return n_occ + 3             # AdaptiveBands at T = 0 (nbands_algorithm.jl:57-66)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "MEASURED_PEAKS.json hbm_gbs (driver-measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


DUMP_BYTES = 32 << 20       # all ranks together; a larger Hψ is sampled


def dump_outputs(path, torch, hpsi, rank, world):
    """Save Hψ (M x n_pw complex) as float64 (n, 2) = (real, imag) rows of the band-major flattened array: all of it when
    it fits DUMP_BYTES / world, else the same seeded sample of entries (seed 0, increasing order) on every run.  Rank r > 0
    of a multi-GPU run writes hpsi_rank<r>.npy."""
    os.makedirs(path, exist_ok=True)
    flat = torch.view_as_real(hpsi).reshape(-1, 2)
    n_keep = min(flat.shape[0], DUMP_BYTES // world // 16)
    if n_keep < flat.shape[0]:
        idx = np.sort(np.random.default_rng(0).choice(flat.shape[0], n_keep, replace=False))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    np.save(os.path.join(path, "hpsi.npy" if rank == 0 else f"hpsi_rank{rank}.npy"), flat.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        self.rows, self.proc = [], None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm))


# ---------------------------------------------------------------------------------------------- oracle arm
def oracle_block(name, n_sample_bands, threads):
    """CPU port of the reference path for the same workload (bounded number of bands)."""
    from oracle.basis import Element, Model, PlaneWaveBasis as OBasis
    from oracle.terms import Terms, energy_hamiltonian, guess_density
    w = WORKLOADS[name]
    lat, pos = supercell(w["rep"])
    om = Model(lat, [Element("Si")] * len(pos), pos, functionals=("lda_x", "lda_c_pw"), symmetries=False,
               terms=("Kinetic", "AtomicLocal", "AtomicNonlocal", "Hartree", "Xc"))
    ob = OBasis(om, w["Ecut"], kcoords=[[0, 0, 0]], kweights=[1.0])
    _, ham = energy_hamiltonian(ob, Terms(ob), None, None, guess_density(ob))
    blk = ham[0]
    blk.workers = threads
    rng = np.random.default_rng(42)
    psi = rng.standard_normal((blk.kpt.n_G, n_sample_bands)) + 1j * rng.standard_normal((blk.kpt.n_G, n_sample_bands))
    return ob, blk, psi


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = effective_cpus()
    os.environ.setdefault("OMP_NUM_THREADS", str(threads))
    nb = min(args.cpu_bands, max(16, 384 // (args.steps + args.warmup)))     # bounded sample: the whole run stays within minutes
    t0 = time.time()
    ob, blk, psi = oracle_block(args.workload, nb, threads)
    setup = time.time() - t0
    for _ in range(args.warmup):
        blk.matmul(psi)
    ts = []
    for _ in range(args.steps):
        t = time.perf_counter()
        blk.matmul(psi)
        ts.append(time.perf_counter() - t)
    dt = sum(ts)
    value = nb * args.steps / dt
    line = dict(metric="hpsi_band_applies_per_s", value=value, unit="band-applies/s", impl="reference", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOADS[args.workload]["desc"], fft_size=list(ob.fft_size), n_pw=int(blk.kpt.n_G),
                            n_proj=int(blk.PD[0].shape[1]), bands_per_step=nb),
                cpu_baseline=dict(value=value, unit="band-applies/s", cores=threads, kind="port",
                                  sample=f"{nb} bands of the {args.workload} block per step (NumPy/pocketfft band loop threaded "
                                         f"over bands + OpenBLAS ZGEMM), oracle restatement of DFTK's CPU path; Julia absent"),
                e2e=dict(value=value, unit="band-applies/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                setup_s=setup)
    print(json.dumps(line), flush=True)



# ---------------------------------------------------------------------------------------------- BASELINE configs C4 / C5
GOLDEN = os.path.join(ROOT, "tests", "golden", "baseline_configs.json")


def baseline_model(dftk, name):
    """BASELINE.json configs[3] / [4] (SURVEY §8d fixes T = 0.01 Ha Fermi-Dirac and Kerker mixing for the metals)."""
    if name == "C5":
        lat = 2.71176 * np.array([[-1, 1, 1], [1, -1, 1], [1, 1, -1]], dtype=float)
        Fe = dftk.ElementPsp("Fe", functional="pbe")
        model = dftk.model_DFT(lat, [Fe], [np.zeros(3)], functionals=dftk.PBE(), temperature=0.01, magnetic_moments=[4.0])
        return model, dict(Ecut=45.0, kgrid=(8, 8, 8)), "Fe bcc PBE collinear spin, Ecut 45 Ha, k 8x8x8 (spin x k blocks sharded)"
    if name == "C4":
        a = 7.65339
        pos = [[0, 0, 0], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]]
        Al = dftk.ElementPsp("Al", functional="pbe")
        model = dftk.model_DFT(a * np.eye(3), [Al] * 4, pos, functionals=dftk.PBE(), temperature=0.01)
        return model, dict(Ecut=40.0, kgrid=(12, 12, 12)), "Al fcc 4-atom PBE, Fermi-Dirac T = 0.01 Ha, Ecut 40 Ha, k 12x12x12 (k blocks sharded)"
    if name == "C2":
        a = 5.131570667152971          # the reference's test lattice (test/testcases.jl:12), the cell of the oracle golden
        lat = np.array([[0, a, a], [a, 0, a], [a, a, 0]])
        Si = dftk.ElementPsp("Si")
        model = dftk.model_DFT(lat, [Si, Si], [np.ones(3) / 8, -np.ones(3) / 8], functionals=dftk.LDA())
        return model, dict(Ecut=30.0, kgrid=(8, 8, 8)), "Si 2-atom LDA, Ecut 30 Ha, k 8x8x8"
    raise KeyError(name)


def sharded_scf(dftk, torch, dist, name, arch, comm, world, dev, repeats=2):
    """A full SCF of a BASELINE config with its (k, spin) blocks sharded over the ranks (STRONG scaling: the total work is
    fixed).  Per step: one NCCL allgather (eigenvalues) + one allreduce (density with the packed energy sums) + the
    converged flag.  Reports the SCF-iteration time (max over ranks) and the energy against the CPU oracle's golden value
    of the same full-size configuration (tests/golden/baseline_configs.json, scripts/make_golden_configs.py)."""
    model, bk, desc = baseline_model(dftk, name)
    t0 = time.perf_counter()
    basis = dftk.PlaneWaveBasis(model, architecture=arch, comm_kpts=comm, **bk)
    setup = time.perf_counter() - t0
    mixing = dftk.KerkerMixing() if model.temperature > 0 else None
    ctx = arch.ctx
    out = None
    for rep in range(repeats):           # the first run warms workspaces / handles
        steps = []
        c0, l0 = comm.n_collectives, ctx.launch_count(reset=True)
        ctx.sync_count(reset=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = time.perf_counter()
        res = dftk.self_consistent_field(basis, tol=1e-8, mixing=mixing, callback=lambda info: steps.append(info["time_step"]), seed=3)
        torch.cuda.synchronize()
        total = time.perf_counter() - t
        tt = torch.tensor([total] + steps, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        tt = tt.cpu().numpy()
        n_it = res["n_iter"]
        out = dict(config=desc, n_ranks=world, fft_size=list(basis.fft_size), blocks_total=basis.layout.n_blocks,
                   blocks_this_rank=len(basis.kpoints), n_bands=int(res["psi"][0].shape[0]), total_s=float(tt[0]), n_iter=n_it,
                   s_per_iter=float(tt[0]) / n_it, step_seconds=[float(x) for x in tt[1:]], converged=bool(res["converged"]),
                   energy=float(res["energies"].total), eF=float(res["eF"]),
                   collectives_per_step=(comm.n_collectives - c0) / n_it if world > 1 else 0,
                   launches_per_step_rank0=ctx.launch_count() / n_it, host_syncs_lobpcg_per_step_rank0=ctx.sync_count() / n_it,
                   setup_s=setup)
    if os.path.exists(GOLDEN):
        g = json.load(open(GOLDEN)).get(name)
        if g:
            n_at = len(model.atoms)
            out["golden_energy"] = g["energies"]["total"]
            out["dE_per_atom_vs_oracle"] = abs(out["energy"] - g["energies"]["total"]) / n_at
            out["d_eF_vs_oracle"] = abs(out["eF"] - g["eF"])
            ev = res["eigenvalues_global"]
            nb = g["n_bands_compared"]
            # the oracle's k-point list may be ordered differently: match blocks by (spin, coordinate)
            dmax = 0.0
            for b in range(basis.layout.n_blocks):
                ik, sp = b % len(basis.kcoords_global), b // len(basis.kcoords_global)
                for j, (kc, s2) in enumerate(zip(g["kcoords"], g["spins"])):
                    if s2 == sp and np.allclose(kc, basis.kcoords_global[ik], atol=1e-10):
                        dmax = max(dmax, float(np.abs(np.asarray(ev[b][:nb]) - np.asarray(g["eigenvalues"][j][:nb])).max()))
                        break
            out["max_d_eigenvalue_vs_oracle"] = dmax
            out["parity_ok"] = bool(out["dE_per_atom_vs_oracle"] < 1e-8 and dmax < 1e-6)
    del basis, res
    torch.cuda.empty_cache()
    return out


def library_gpu_baseline(torch, basis, blk, kb, psi, n_local_bands):
    """The reference's GPU formulation of H psi with LIBRARY kernels (what ext/DFTKCUDAExt.jl gets from cuFFT + cuBLAS,
    src/terms/Hamiltonian.jl:155-176 + src/fft.jl:110-172): band at a time zero-fill, scatter, cuFFT backward, multiply,
    cuFFT forward, gather, kinetic axpy; nonlocal term as two cuBLAS ZGEMMs.  Timed with CUDA events on the same block."""
    dev = psi.device
    nx, ny, nz = basis.fft_size
    N = basis.N
    mapping = basis.kpoints[blk.ik].mapping
    V = blk.local_op.potential.reshape(nz, ny, nx)
    kin = blk.fourier_op.multiplier
    P = blk.nonlocal_op.P                               # (n_proj, n_pw) = column-major n_pw x n_proj
    D = torch.as_tensor(blk.nonlocal_op.D, device=dev, dtype=torch.complex128)
    cube = torch.empty(N, dtype=torch.complex128, device=dev)
    nb = min(n_local_bands, psi.shape[0])
    out = torch.empty((nb, psi.shape[1]), dtype=torch.complex128, device=dev)

    def local(n_bands):
        for n in range(n_bands):
            cube.zero_()
            cube[mapping] = psi[n]
            r = torch.fft.ifftn(cube.view(nz, ny, nx))          # includes the 1/N of fft_norm * ifft_norm
            r.mul_(V)
            f = torch.fft.fftn(r)
            out[n] = f.view(-1)[mapping] + kin * psi[n]

    def nonlocal_(x):
        proj = torch.conj(P) @ x.T                              # P' psi   (n_proj x M)
        return (P.T @ (D @ proj)).T

    def ev(fn, reps=2):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    ms_local = ev(lambda: local(nb)) / nb                        # per band
    ms_nl = ev(lambda: nonlocal_(psi))                           # whole block
    M = psi.shape[0]
    # correctness of the formulation against the product on the sampled bands
    local(min(nb, 4))
    hp = out[:min(nb, 4)] + nonlocal_(psi[:min(nb, 4)])
    ref = kb.apply_h(psi[:min(nb, 4)].contiguous())
    err = float((hp - ref).abs().max() / ref.abs().max())
    ms_block = ms_local * M + ms_nl
    return dict(value=M / (ms_block * 1e-3), unit="band-applies/s", ms_per_block=ms_block, us_per_band_local=1e3 * ms_local,
                ms_nonlocal=ms_nl, bands_sampled_local=nb, max_rel_diff_vs_product=err,
                what="band-at-a-time zero-fill + scatter + cuFFT Z2Z + multiply + cuFFT + gather + axpy (torch.fft) and two cuBLAS "
                     "ZGEMMs (torch.matmul) on the same block: the reference's own GPU formulation with library kernels")


# ---------------------------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    # Keep stdout clean for the single JSON line: C libraries (e.g. the NCCL version banner) write to fd 1.
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    # (thread pools were sized at import time: torchrun's OMP_NUM_THREADS=1 starves cuSOLVER's heevd host stages,
    #  an unset value oversubscribes CPU-quota containers)
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    import dftk_b200 as dftk
    comm = dftk.KpointComm.from_torch_distributed() if world > 1 else dftk.KpointComm()
    arch = dftk.B200(local, comm=comm if world > 1 else None)
    ctx, dev = arch.ctx, arch.device
    w = WORKLOADS[args.workload]
    lat, pos = supercell(w["rep"])
    t0 = time.time()
    Si = dftk.ElementPsp("Si")
    model = dftk.model_DFT(lat, [Si] * len(pos), pos, functionals=dftk.LDA(), symmetries=False)
    # one k-block per rank: Gamma plus distinct shifted k-points for the other ranks (same N_pw to ~0.1 %)
    kcoords = [[0.0, 0.0, 0.0]] + [[0.5 * (i % 2), 0.5 * ((i // 2) % 2), 0.5 * ((i // 4) % 2)] for i in range(1, world)]
    basis = dftk.PlaneWaveBasis(model, Ecut=w["Ecut"], kgrid=dftk.ExplicitKpoints(kcoords), architecture=arch,
                                comm_kpts=comm)
    rho0 = dftk.guess_density(basis)
    energies0, ham = dftk.energy_hamiltonian(basis, None, None, rho=rho0)
    blk = ham[0]
    kb = blk.bind()
    n_pw, N = kb.n_pw, basis.N
    M = args.bands or n_bands_for(len(pos))
    setup = time.time() - t0
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    psi = torch.view_as_complex(torch.randn(M, n_pw, 2, generator=g, device=dev, dtype=torch.float64))
    hpsi = torch.empty_like(psi)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- headline: full H apply on device-resident data
    sampler = ClockSampler(local) if rank == 0 else None
    ctx.launch_count(reset=True)
    ms_total = timed(lambda: kb.apply_h(psi, hpsi), args.steps, args.warmup)
    launches = ctx.launch_count() // max(1, 1)    # launches since reset (includes warm-up)
    launches_timed = int(round(launches * args.steps / (args.steps + args.warmup)))
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    value = world * M * args.steps / (ms_total * 1e-3)
    if args.dump_outputs:           # before the sections below overwrite hpsi
        dump_outputs(args.dump_outputs, torch, hpsi, rank, world)

    # ---- kernel-group breakdown (same stream, CUDA events)
    ms_local = timed(lambda: kb.apply_terms(psi, 3, out=hpsi), max(2, args.steps // 2), 1) / max(2, args.steps // 2)
    ms_nl = timed(lambda: kb.apply_terms(psi, 4, out=hpsi), max(2, args.steps // 2), 1) / max(2, args.steps // 2)
    hbm_peak, peak_src = peaks()
    alg_bytes_band = 72.0 * N + 40.0 * n_pw
    ach = alg_bytes_band * M / (ms_local * 1e-3) / 1e9
    # measured DRAM traffic of the group (dram__bytes_read.sum + dram__bytes_write.sum over the five kernels of one
    # `ncu --set full` capture, profiles/ncu_full_r1.csv: 17.11 GB per 51-band launch on the 192^3 grid), scaled to the
    # block like `achieved`; only known for the profiled workload
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")       # written by scripts/summarize_ncu.py from the round's
    if args.workload == "si250" and os.path.exists(tpath):            # `ncu --set full` capture (dram bytes read + written)
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["hpsi_local_dram_bytes_per_band"] * M, tj["source"]
    roofline = dict(bound="hbm", kernel="Hpsi-local group (kr_sphere_to_x, kr_y_backward, kr_z_apply, kr_y_forward, kr_x_to_sphere)",
                    achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, traffic=traffic,
                    traffic_source=traffic_src,
                    algorithmic_bytes_per_band=alg_bytes_band, ms_per_block=ms_local, us_per_band=1e3 * ms_local / M,
                    peak_source=peak_src + " (of measured)")
    n_proj = kb.n_proj
    fl_nl = 16.0 * n_pw * n_proj * M
    # the same two projector products on the FP64 DMMA pipe: own kernels (gemm_backend 0) and cuBLAS ZGEMM (gemm_backend 1, the
    # FP64 peak calibration; MEASURED_PEAKS.json has no FP64 figure).  The default path (gemm_backend 4) runs them on the INT8
    # tensor cores (tcgen05.mma.kind::i8, exact FP64-equivalent results through residues + CRT), so `frac` can exceed 1.
    backend_default = 4
    ctx.set_option("gemm_backend", 1)
    ms_nl_cublas = timed(lambda: kb.apply_terms(psi, 4, out=hpsi), 2, 1) / 2
    ctx.set_option("gemm_backend", 0)
    ms_nl_dmma = timed(lambda: kb.apply_terms(psi, 4, out=hpsi), 2, 1) / 2
    ctx.set_option("gemm_backend", backend_default)
    tf_nl, tf_cublas, tf_dmma = (fl_nl / (t * 1e-3) / 1e12 for t in (ms_nl, ms_nl_cublas, ms_nl_dmma))
    roofline_gemm = dict(bound="tensor", kernel="nonlocal P D P'psi: k_i8_gemm_tc2 + k_i8_gemm_tc2_nn (tcgen05.mma.kind::i8, TMA-fed, INT8 residues + CRT) "
                                                "with k_i8_residues_ld4 / k_i8_crt_nn around them",
                         achieved=tf_nl, peak=tf_cublas, unit="TFLOP/s (FP64-equivalent)", frac=tf_nl / tf_cublas, flop=fl_nl, ms=ms_nl,
                         peak_source="cuBLAS ZGEMM (FP64 DMMA pipe) on the same shapes in the same run; nominal FP64 tensor 37-40 TFLOP/s",
                         own_dmma_kernels=dict(ms=ms_nl_dmma, achieved=tf_dmma, frac_of_cublas=tf_dmma / tf_cublas, frac_of_fixed_36TF=tf_dmma / 36.0),
                         tensor_pipe_evidence="profiles/ncu_i8_r2.csv: sm__pipe_tensor_cycles_active of k_i8_gemm_tc2 / k_i8_gemm_tc2_nn")
    # ---- the reference's GPU formulation with library kernels (cuFFT band-at-a-time + cuBLAS) on the same block
    lib_gpu = None
    if rank == 0 and not args.no_library:
        try:
            lib_gpu = library_gpu_baseline(torch, basis, blk, kb, psi, 32)
            lib_gpu["speedup_of_product"] = (M / (ms_step * 1e-3)) / lib_gpu["value"]
        except Exception as e:
            lib_gpu = dict(error=repr(e))

    # ---- end to end through the C ABI with pinned host buffers
    e2e = None
    if not args.no_e2e:
        from dftk_b200._lib import check
        from dftk_b200.device import _ptr
        hpsi_h = torch.empty((M, n_pw), dtype=torch.complex128, pin_memory=True)
        psi_h = torch.empty((M, n_pw), dtype=torch.complex128, pin_memory=True)
        psi_h.copy_(psi)

        def e2e_step():
            check(ctx.L.dftk_b200_apply_h(kb.h, _ptr(psi_h), _ptr(hpsi_h), M), ctx.h)
        ksteps = max(1, min(args.steps, 3))
        for _ in range(1):
            e2e_step()
        barrier()
        t = time.perf_counter()
        for _ in range(ksteps):
            e2e_step()
        barrier()
        dt = time.perf_counter() - t
        if world > 1:
            tt = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        nbytes = M * n_pw * 16
        e2e = dict(value=world * M * ksteps / dt, unit="band-applies/s", h2d_bytes_per_step=nbytes, d2h_bytes_per_step=nbytes,
                   ms_per_step=1e3 * dt / ksteps)
        del psi_h, hpsi_h

    # ---- density accumulate + allreduce (the one real collective of an SCF step)
    extra = {}
    occ_w = np.full(M, 2.0)
    rho = torch.zeros(N, dtype=torch.float64, device=dev)
    ms_rho = timed(lambda: kb.density_accumulate(psi, occ_w, rho), 2, 1) / 2
    extra["density_ms_per_block"] = ms_rho
    extra["density_GBs_alg"] = (32.0 * N + 16.0 * n_pw) * M / (ms_rho * 1e-3) / 1e9
    if world > 1:
        rbuf = torch.zeros((1, N), dtype=torch.float64, device=dev)
        extra["rho_allreduce_ms"] = timed(lambda: ctx.allreduce(rbuf), 5, 2) / 5
    # ---- one LOBPCG solve at loose tolerance = the eigensolver part of the first SCF step (optional)
    if args.scf:
        X = psi.clone()
        kb.lobpcg(X, tol=args.scf_tol, maxiter=1, n_conv_check=M - 3)   # untimed: cuSOLVER handles, 23 GB workspace
        X.copy_(psi)
        torch.cuda.synchronize()
        try:
            ctx.lobpcg_flops(reset=True)
        except Exception:
            pass
        t = time.perf_counter()
        res = kb.lobpcg(X, tol=args.scf_tol, maxiter=args.scf_maxiter, n_conv_check=M - 3)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        extra["lobpcg"] = dict(seconds=dt, n_iter=res["n_iter"], n_matvec=res["n_matvec"], converged=res["converged"],
                               tol=args.scf_tol, s_per_iter=dt / max(1, res["n_iter"]))
        try:
            fl = ctx.lobpcg_flops(reset=True)
            extra["lobpcg"].update(gemm_flop=fl, gemm_TFLOPs_fp64_equivalent=fl / dt / 1e12,
                                   note="GEMM flops executed (Gram, update, Cholesky-QR and nonlocal products, counted in the library) over "
                                        "the WHOLE solve time, which also contains the FFT part of H, the eigensolver and host syncs")
        except Exception as e:
            extra["lobpcg"]["gemm_flop_error"] = repr(e)
        del X

    # ---- single-k multi-GPU (SURVEY §8 f3): the SAME Gamma block solved by all ranks together (plane-wave slabs: local Gram
    #      products + NCCL allreduce, rows <-> bands exchange around H) against one GPU solving it alone, same start vectors
    if world > 1 and args.scf and not args.no_slab:
        try:
            kb.trim()        # the 503-band solve above left ~60 GB of solver scratch on this rank's k-block
            torch.cuda.empty_cache()
            bs = dftk.PlaneWaveBasis(model, Ecut=w["Ecut"], kgrid=(1, 1, 1), architecture=arch, comm_slab=comm)
            hs = dftk.energy_hamiltonian(bs, None, None, rho=dftk.guess_density(bs))[1]
            kbs = hs[0].bind()
            gs = torch.Generator(device=dev).manual_seed(4242)
            X0 = torch.view_as_complex(torch.randn(M, kbs.n_pw, 2, generator=gs, device=dev, dtype=torch.float64))
            X = X0.clone()
            out = {}
            for name, solve in (("slab", kbs.lobpcg_slab), ("one_gpu", kbs.lobpcg)):
                # untimed first pass: workspaces, residue-plane pools of all blocks (P / AP appear from the 2nd iteration),
                # cuSOLVER handles, NCCL point-to-point connections
                solve(X, tol=args.scf_tol, maxiter=args.scf_maxiter, n_conv_check=M - 3)
                X.copy_(X0)
                barrier()
                dist.barrier()
                t = time.perf_counter()
                r = solve(X, tol=args.scf_tol, maxiter=args.scf_maxiter, n_conv_check=M - 3)
                torch.cuda.synchronize()
                dt = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
                out[name] = dict(seconds=float(dt.item()), n_iter=r["n_iter"], s_per_iter=float(dt.item()) / max(1, r["n_iter"]),
                                 lam=r["λ"].copy(), exchange_GB=r.get("exchange_bytes", 0.0) / 1e9)
            dl = float(np.abs(out["slab"]["lam"] - out["one_gpu"]["lam"]).max())
            for v in out.values():
                del v["lam"]
            extra["single_k_slab"] = dict(n_ranks=world, n_pw=int(kbs.n_pw), n_bands=M, slab=out["slab"], one_gpu=out["one_gpu"],
                                          speedup_vs_one_gpu=out["one_gpu"]["s_per_iter"] / out["slab"]["s_per_iter"],
                                          max_dlambda_vs_one_gpu=dl,
                                          what="LOBPCG on ONE k-point (C3 Gamma block) by all ranks: plane-wave slabs, Gram "
                                               "products completed by ncclAllReduce, H applied band-wise after a rows<->bands exchange")
            del X, X0
            kbs.trim()       # scratch of the one-GPU comparison solve
            torch.cuda.empty_cache()
            # real SCF iterations of the SAME single-k-point cell with all ranks on it (slab eigensolver, band-shared density,
            # one density/energy allreduce per step): compare with the `scf` key of the N = 1 line
            if args.scf_steps > 0 or args.slab_scf_steps > 0:
                st, it = [], []

                def cbs(info):
                    st.append(info["time_step"])
                    it.append(int(np.sum(info["diagonalization"]["n_iter"])))
                c0 = comm.n_collectives
                tq = time.perf_counter()
                rs = dftk.self_consistent_field(bs, tol=1e-10, maxiter=max(args.scf_steps, args.slab_scf_steps), callback=cbs, seed=1)
                torch.cuda.synchronize()
                extra["single_k_slab"]["scf"] = dict(step_seconds=st, lobpcg_iters_per_step=it, total_s=time.perf_counter() - tq,
                                                     energy_per_atom=rs["energies"].total / len(pos), last_drho=rs["history_drho"][-1],
                                                     collectives_per_step=(comm.n_collectives - c0) / max(1, rs["n_iter"]),
                                                     note="same cell, tolerances and seed as the `scf` key of the N = 1 line")
                del rs
            del bs, hs, kbs
            torch.cuda.empty_cache()
        except Exception as e:
            extra["single_k_slab"] = dict(error=repr(e))
            if world > 1:
                raise       # a rank that left a collective solve early would hang the others: fail loudly instead

    # ---- real SCF iterations on this workload (energy_hamiltonian + LOBPCG + occupations + density [+ allreduce]
    #      + consistent energies + mixing): the "SCF iteration time" half of the metric
    if args.scf_steps > 0:
        del psi, hpsi
        torch.cuda.empty_cache()
        scf_t, scf_it = [], []

        def cb(info):
            scf_t.append(info["time_step"])
            scf_it.append(int(np.sum(info["diagonalization"]["n_iter"])))
        t = time.perf_counter()
        res = dftk.self_consistent_field(basis, tol=1e-10, maxiter=args.scf_steps, callback=cb, seed=1)
        torch.cuda.synchronize()
        extra["scf"] = dict(step_seconds=scf_t, lobpcg_iters_per_step=scf_it, total_s=time.perf_counter() - t,
                            energy_per_atom=res["energies"].total / len(pos), last_drho=res["history_drho"][-1],
                            note="step 1 starts from random orbitals (loose AdaptiveDiagtol tolerance), later steps from the previous orbitals")
        # ---- Hellmann-Feynman forces of that state (SURVEY §8f rank 4): local (one cube pass per atom), nonlocal (four
        #      DMMA projections per k-block), Ewald (host)
        try:
            if world > 1:
                raise RuntimeError("measured at N=1 only")
            from dftk_b200 import forces as fmod
            ft = {}
            for name, fn in (("local", lambda: fmod.forces_local(basis, res["rho"])),
                             ("nonlocal", lambda: fmod.forces_nonlocal(basis, res["psi"], res["occupation"]))):
                fn()
                torch.cuda.synchronize()
                t = time.perf_counter()
                f = fn()
                torch.cuda.synchronize()
                ft[name + "_s"] = time.perf_counter() - t
                ft[name + "_max_abs"] = float(np.abs(np.array(f)).max())
            fmod.energy_forces_ewald_device(ctx, lat, [4.0] * len(pos), pos)
            t = time.perf_counter()
            fmod.energy_forces_ewald_device(ctx, lat, [4.0] * len(pos), pos)
            ft["ewald_device_s"] = time.perf_counter() - t
            nbf = int(np.count_nonzero(res["occupation"][0]))
            ft["nonlocal_TFLOPs"] = 4 * 8.0 * n_pw * kb.n_proj * nbf / ft["nonlocal_s"] / 1e12
            extra["forces"] = ft
        except Exception as e:      # never lose the headline line to the optional section
            extra["forces"] = dict(error=repr(e))
        psi = torch.view_as_complex(torch.randn(M, n_pw, 2, generator=g, device=dev, dtype=torch.float64))
        kb.set_potential(blk.local_op.potential)     # the SCF installed its own potentials; restore the benchmark operator

    # ---- BASELINE config C2 (Si2 LDA, Ecut 30, 8x8x8 k-grid: 29 irreducible k-blocks of 7 bands) -- a full SCF to 1e-8;
    #      the launch-latency-bound regime (fused small-matrix LOBPCG kernels), reported beside the C3 numbers
    if args.scf_steps > 0 and world == 1 and not args.no_small:
        try:
            m2, bk2, _ = baseline_model(dftk, "C2")
            b2 = dftk.PlaneWaveBasis(m2, architecture=arch, **bk2)
            dftk.self_consistent_field(b2, tol=1e-8)            # warm-up (workspaces, cuSOLVER handles)
            torch.cuda.synchronize()
            ctx.launch_count(reset=True)
            ctx.sync_count(reset=True)
            t = time.perf_counter()
            r2 = dftk.self_consistent_field(b2, tol=1e-8)
            torch.cuda.synchronize()
            dt2 = time.perf_counter() - t
            l2, s2 = ctx.launch_count(), ctx.sync_count()
            extra["scf_c2"] = dict(total_s=dt2, n_iter=r2["n_iter"], s_per_iter=dt2 / r2["n_iter"], k_blocks=len(b2.kpoints),
                                   fft_size=list(b2.fft_size), energy=r2["energies"].total, converged=bool(r2["converged"]),
                                   launches_per_scf_step=l2 / r2["n_iter"], lobpcg_host_syncs_per_scf_step=s2 / r2["n_iter"])
            if os.path.exists(GOLDEN) and "C2" in json.load(open(GOLDEN)):
                g2 = json.load(open(GOLDEN))["C2"]
                extra["scf_c2"]["dE_per_atom_vs_oracle"] = abs(r2["energies"].total - g2["energies"]["total"]) / 2
            del b2, r2
        except Exception as e:
            extra["scf_c2"] = dict(error=repr(e))

    # ---- BASELINE configs C5 / C4: full SCFs with the (k, spin) blocks sharded over the ranks (strong scaling, parity vs
    #      the oracle's golden energies asserted in the line)
    if not args.no_sharded:
        sh = {}
        for name in args.sharded.split(","):
            try:
                sh[name] = sharded_scf(dftk, torch, dist, name, arch, comm, world, dev)
            except Exception as e:
                sh[name] = dict(error=repr(e))
        extra["sharded_scf"] = sh

    # ---- CPU baseline on rank 0 (bounded sample)
    cpu = None
    if rank == 0 and not args.no_cpu:
        threads = effective_cpus()
        nb = args.cpu_bands
        P = kb_P = None
        from oracle.terms import HamiltonianBlock
        from oracle.basis import Kpoint as OKpoint

        class _B:      # minimal oracle-basis view over the same operator data (fft methods only)
            pass
        from oracle.basis import PlaneWaveBasis as OBasis, Model as OModel, Element
        om = OModel(lat, [Element("Si")] * len(pos), pos, symmetries=False, terms=("Kinetic",))
        ob = OBasis(om, w["Ecut"], kcoords=[[0, 0, 0]], kweights=[1.0])
        blk0_kin = basis.term("Kinetic").kinetic_energies[0].cpu().numpy()
        V = blk.local_op.potential.cpu().numpy()
        nlop = basis.term("AtomicNonlocal").ops[0]
        Pn = nlop.P.cpu().numpy().T.copy() if rank == 0 else None
        oblk = HamiltonianBlock(ob, 0, blk0_kin, V, (Pn, nlop.D))
        oblk.workers = threads
        xs = psi[:nb].cpu().numpy().T.copy()
        oblk.matmul(xs[:, :1])
        t = time.perf_counter()
        ref = oblk.matmul(xs)
        dt = time.perf_counter() - t
        got = hpsi_check = kb.apply_h(psi[:nb].contiguous()).cpu().numpy().T
        err = float(np.abs(got - ref).max() / np.abs(ref).max())
        # single-thread number (the reference's own benchmark protocol, benchmark/run_benchmarks.jl:86)
        oblk.workers = 1
        try:
            from threadpoolctl import threadpool_limits
            with threadpool_limits(limits=1):
                t = time.perf_counter()
                oblk.matmul(xs[:, :2])
                dt1 = time.perf_counter() - t
        except Exception:
            t = time.perf_counter()
            oblk.matmul(xs[:, :2])
            dt1 = time.perf_counter() - t
        oblk.workers = threads
        # the reference's rule of thumb (docs/src/tricks/parallelization.md:62-72): 30 ms per 128^3 FFT and thread, two FFTs
        # per band apply (FFT part only; the nonlocal GEMMs come on top)
        rot = 2 * 0.030 * N / 128 ** 3
        cpu = dict(value=nb / dt, unit="band-applies/s", cores=threads, kind="port",
                   sample=f"{nb} bands of the same block, one pass (NumPy pocketfft band loop threaded over bands + OpenBLAS ZGEMM)",
                   seconds=dt, max_rel_err_vs_gpu=err,
                   single_thread=dict(value=2 / dt1, unit="band-applies/s", cores=1, sample="2 bands of the same block, one thread"),
                   reference_rule_of_thumb=dict(seconds_per_band_per_thread_fft_only=rot, value_all_cores=threads / rot, unit="band-applies/s",
                                                source="docs/src/tricks/parallelization.md:62-72 (30 ms per 128^3 FFT per thread, 2 FFTs per band)"))
        del Pn

    parity = dict(tolerances="energy 1e-8 Ha/atom, eigenvalues 1e-6 Ha (BASELINE.json north_star)",
                  c3_hpsi_max_rel_err_vs_oracle=(cpu or {}).get("max_rel_err_vs_gpu"),
                  c2_dE_per_atom_vs_oracle=extra.get("scf_c2", {}).get("dE_per_atom_vs_oracle"),
                  **{f"{k.lower()}_dE_per_atom_vs_oracle": v.get("dE_per_atom_vs_oracle") for k, v in extra.get("sharded_scf", {}).items()},
                  **{f"{k.lower()}_max_d_eigenvalue_vs_oracle": v.get("max_d_eigenvalue_vs_oracle") for k, v in extra.get("sharded_scf", {}).items()})
    if rank == 0:
        line = dict(metric="hpsi_band_applies_per_s", value=value, unit="band-applies/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f64", data="synthetic",
                    config=dict(workload=w["desc"] + (f", one k-block per GPU ({world} k-points)" if world > 1 else ""),
                                fft_size=list(basis.fft_size), n_pw=n_pw, n_bands=M, n_proj=n_proj,
                                parallelism=f"kpoints x{world}", cache="inputs (psi 16*n_pw*M bytes) larger than L2"),
                    block_applies_per_s=world * args.steps / (ms_total * 1e-3),
                    roofline=roofline, roofline_gemm=roofline_gemm, cpu_baseline=cpu, gpu_library_baseline=lib_gpu, e2e=e2e,
                    gpu_launches=launches_timed, parity=parity,
                    clocks=clocks, setup_s=setup, **extra)
        os.write(saved_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DFTK_BENCH_WORKLOAD", "si250"), choices=list(WORKLOADS))
    ap.add_argument("--bands", type=int, default=0)
    ap.add_argument("--cpu-bands", type=int, default=0,
                    help="bands in the CPU sample (0 = 64)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-library", action="store_true", help="skip the cuFFT/cuBLAS formulation of the same H apply")
    ap.add_argument("--no-small", action="store_true", help="skip the full SCF of BASELINE config C2")
    ap.add_argument("--no-slab", action="store_true", help="skip the single-k multi-GPU (plane-wave slab) LOBPCG section at N > 1")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded SCFs of the BASELINE metal configs")
    ap.add_argument("--sharded", default="C5,C4", help="BASELINE configs whose (k, spin) blocks are sharded over the ranks")
    ap.add_argument("--no-scf", dest="scf", action="store_false",
                    help="skip the LOBPCG timing (eigensolver part of an SCF step, a few iterations)")
    ap.set_defaults(scf=True)
    ap.add_argument("--scf-steps", type=int, default=3, help="real SCF iterations to time (0 = skip)")
    ap.add_argument("--slab-scf-steps", type=int, default=0, help="SCF iterations of the single-k slab section when --scf-steps is 0")
    ap.add_argument("--scf-tol", type=float, default=0.025)
    ap.add_argument("--scf-maxiter", type=int, default=6)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write H psi of the last timed step to DIR/hpsi.npy (float64 real/imag pairs, seeded sample when large)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    if args.cpu_bands <= 0:
        args.cpu_bands = 64      # enough columns for the CPU ZGEMM not to be bound by the bandwidth of P
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
