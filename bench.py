#!/usr/bin/env python
"""
bench.py -- NUTS leapfrog-steps x chains / s, cubic-2 PolyModel surrogate, d=26 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one complete NUTS run (n_iter=1500, n_warmup=500: reference defaults, sample_trace.py:499-512)
of 4096 chains per GPU on the 26-D DES-Y1-shaped synthetic posterior (SURVEY.md 8d config 3 = BASELINE.json
configs[2]: 32768 chains over 8 GPUs) through its fitted cubic-2 surrogate: ONE kernel launch (+ device-side reset of
the chain state).  Weak scaling: every rank runs its own 4096 chains (global chain ids -> distinct Philox streams), no
data-path collective.  The dominant kernel is nuts_dmma_kernel (bfb_sampler_dmma.cu: 8 chains per warp as the rows of
FP64 m8n8k4 DMMAs).  4096 chains are 512 warps -- fewer than the 592 warp schedulers of a B200 -- so the line also
carries `more_chains` (north_star: "at least 4096 chains per GPU"): the same run with 16384 chains on this GPU, and
`eval_kernel`: the batched surrogate evaluation kernel alone (bfb_eval_dmma.cu) against the same FP64 peak.
`pipeline_kernel`: SURVEY 8f rank 1 -- DES-Y1-shaped surrogate -> Gaussian-likelihood pipeline (n = 26, m = 457 outputs) on the
tensor cores: batched logp + gradient (bfb_lik_dmma.cu) and a 4096-chain NUTS run (model variant bit 3), same FP64 peak.

  value : sum(tree_size) of all ranks / max-over-ranks device time of K steps, inputs resident in HBM
  e2e   : the same through bayesfast_b200.sample(keep='post_warmup') with host x_0; the samples and all statistics of the
          1000 post-warm-up iterations come back to pinned host memory (what SampleTrace.get hands to its callers,
          sample_trace.py:762-787; the warm-up records never leave the device).  `e2e_variants` (N = 1): every record of every
          iteration (round-1 definition), and thin=10 + on-device mean / covariance.
  roofline : algorithmic FP64 flops (8n^2+24n per chain-leapfrog, SURVEY.md 8d) / kernel time (CUDA events on
             the launching stream) vs the FP64 peak measured in this run (MEASURED_PEAKS.json has no FP64 entry)
  cpu_baseline : the UNMODIFIED reference (baseline/_ref, installed by __graft_entry__.build()) through its own public API
             and multiprocess chain pool (bf.sample + set_backend(cores)) on this box's host cores, full-length chains of the
             same workload; next to it `port`: the oracle (C restatement, OpenMP over chains).  `--impl reference` runs only
             the reference arm (the port when baseline/_ref is missing; the line says which).
  extras (N = 1 unless noted): more_chains, team_kernel, pair_kernel, hmc_kernel, eval_kernel, pipeline_kernel, config3 (64-D cubic-3),
             fit_sweep (d = 32 cubic-2, N = 1e4 .. 1e7 rows; at N > 1 GPUs rows sharded + the NCCL all-reduce timed).
  --dump-outputs DIR : the outputs of the last timed step as DIR/<name>.npy (see dump_outputs), to compare two builds; with
             N > 1 GPUs only rank 0 writes, so the files cover its own chains, 1/N of the step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DIM, ORDER, CHAINS_PER_GPU, N_ITER, N_WARMUP, SEED = 26, 'cubic-2', 4096, 1500, 500, 20261017
FLOPS_PER_LEAF = 8 * N_DIM * N_DIM + 24 * N_DIM        # SURVEY.md 8(d): 6032 at n=26
WORKLOAD = 'des_y1_shaped_d26_cubic2_nuts_4096_chains_per_gpu_n_iter1500_n_warmup500'


def clocks_sampler(stop, out, device):
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    while not stop.is_set():
        try:
            r = subprocess.run(['nvidia-smi', '-i', str(device), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                               capture_output=True, text=True, timeout=5).stdout.strip().split(',')
            out.append([v.strip() for v in r])
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    if not samples:
        return None
    sm = sorted(float(s[0]) for s in samples if s[0].replace('.', '').isdigit())
    names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
    reasons = [nm for i, nm in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower().startswith('active') for s in samples)]
    return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=float(samples[0][1]) if samples[0][1] else None,
                power_w_max=max(float(s[2]) for s in samples if s[2].replace('.', '').isdigit()), reasons=reasons,
                samples=len(samples))


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def oracle_spec_cpu(prob):
    """surrogate fitted on the CPU with the oracle (scipy lstsq), for the reference arm"""
    from oracle import bf_oracle as o
    n = prob['n']
    cfgs = [dict(order=k, input_mask=np.arange(n), output_mask=np.arange(1)) for k in ('linear', 'quadratic', 'cubic-2')]
    coefs = o.fit(cfgs, n, 1, prob['x_fit'], prob['y_fit'])
    for c, a in zip(cfgs, coefs):
        c['coef'] = a
    mu, hess, alpha = o.bound_from_points(prob['x_fit'])
    spec = dict(n=n, m=1, configs=cfgs, use_bound=False, input_scales=None, use_decay=False, transform_ranges=None)
    xm = prob['x_fit'][int(np.argmax(prob['y_fit'][:, 0]))]
    f_mu = o.OracleDensity(spec).poly_eval_batch(xm[None])[0][0]
    spec.update(use_bound=True, mu=mu, hess=hess, alpha=alpha, f_mu=f_mu)
    return spec


def run_cpu_baseline(spec, prob, budget_s=15., n_threads=0):
    """the oracle port on all host cores: bounded sample = as many full chains (n_iter=1500) as fit in ~budget_s"""
    from oracle import bf_oracle as o
    cores = cpu_cores() if n_threads <= 0 else n_threads
    od = o.OracleDensity(spec)
    n = prob['n']
    cfg = dict(n_iter=N_ITER, n_warmup=N_WARMUP, seed=SEED, n_threads=cores)
    step0 = 1. / n**0.25
    t0 = time.time()
    r = od.run('NUTS', cfg, prob['x_0'][:cores], step0, np.ones(n))
    t_probe = time.time() - t0
    chains = int(max(cores, min(prob['x_0'].shape[0], cores * max(1, int(budget_s / max(t_probe, 1e-3))))))
    t0 = time.time()
    r = od.run('NUTS', cfg, prob['x_0'][:chains], step0, np.ones(n))
    dt = time.time() - t0
    leaves = int(r['tree_size'].sum())
    return dict(value=leaves / dt, unit='leapfrog-steps*chains/s', cores=cores, kind='port',
                sample='{} full chains (n_iter={}, n_warmup={}) of the same workload, {} leapfrogs in {:.1f} s, oracle/'
                       'libbf_oracle.so (C restatement, OpenMP over chains); the Python reference itself measured '
                       '3.2e4/s on 8 cores (BASELINE.md)'.format(chains, N_ITER, N_WARMUP, leaves, dt)), leaves, dt


def run_reference_python(prob, cores, per=2, n_iter=N_ITER, n_warmup=N_WARMUP, timeout=900):
    """the real reference (baseline/_ref) in a subprocess: bf.sample over its own process pool; None if it is not installed"""
    import glob
    import tempfile
    if not glob.glob(os.path.join(ROOT, 'baseline', '_ref', 'bayesfast', 'modules', '_poly*.so')):
        return None
    n_chain = cores * per
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, 'in.npz')
        np.savez(f, x_fit=prob['x_fit'], y_fit=prob['y_fit'], x_0=prob['x_0'][:n_chain], n_iter=n_iter, n_warmup=n_warmup, order=ORDER)
        env = dict(os.environ, OMP_NUM_THREADS='1', OPENBLAS_NUM_THREADS='1', MKL_NUM_THREADS='1')
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, 'baseline', 'ref_runner.py'), f, str(cores), str(per)],
                               capture_output=True, text=True, timeout=timeout, env=env)
            out = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as exc:
            return dict(error=repr(exc))
    return dict(value=out['value'], unit='leapfrog-steps*chains/s', cores=cores, kind='reference', leaves=out['leaves'], seconds=out['wall_s'],
                per_core=out['value'] / cores, fit_seconds=out['fit_s'], mean_tree_size=out['mean_tree_size'],
                sample='h3jia/bayesfast unmodified (baseline/_ref): bf.sample, NUTS, set_backend({0}), {1} full chains (n_iter={2}, '
                       'n_warmup={3}) of the same workload, {4} leapfrogs in {5:.1f} s wall including pool start-up'.format(
                           cores, out['n_chain'], n_iter, n_warmup, out['leaves'], out['wall_s']))


def extra_measurements(args, bfb, torch, den, h, prob, x0, trace_kw, flush, peak, dev, C):
    """supplementary numbers of the bench line (rank 0, single GPU): none of them enters `value` / `e2e`"""
    from bayesfast_b200 import synthetic, _cabi
    extras = {}
    # (a) the same run with 16384 chains on this GPU (two warps per scheduler instead of one): kernel-only value
    C2 = 16384
    prob2 = synthetic.des_shaped(N_DIM, seed=1, n_chain=C2, order=ORDER)
    cfg2 = bfb.NTrace(n_chain=C2, n_iter=N_ITER, n_warmup=N_WARMUP, x_0=prob2['x_0'], random_generator=SEED)._cfg_dict(SEED, 0)
    h.sampler_init(cfg2, prob2['x_0'], 1. / N_DIM**0.25, np.ones(N_DIM), prob2['x_0'])
    best = None
    for i in range(3):
        h.sampler_reset()
        flush.zero_()
        torch.cuda.synchronize(dev)
        r2 = h.sampler_run('NUTS', N_ITER, out_ptrs={})
        ms2 = h.last_kernel_ms()
        if i > 0 and (best is None or ms2 < best[1]):
            best = (r2['total_tree_size'], ms2)
    tf2 = FLOPS_PER_LEAF * best[0] / (best[1] * 1e-3) / 1e12
    extras['more_chains'] = dict(chains_per_gpu=C2, value=best[0] / (best[1] * 1e-3), unit='leapfrog-steps*chains/s',
                                 kernel_ms=best[1], outputs='none written (kernel only)', kernel=h.sampler_last_path(),
                                 roofline_frac=tf2 / peak, achieved_tflops=tf2)
    # (a2) lock-step HMC (hmc.py:16-49, n_int_step = 32) on the same chains: the tensor-core integrator without the NUTS
    # tree bookkeeping (hmc_dmma_kernel), kernel only
    hm = {}
    for Ch, x0h in ((C, x0), (C2, prob2['x_0'])):
        cfgh = bfb.HTrace(n_chain=Ch, n_iter=300, n_warmup=100, x_0=x0h, n_int_step=32, random_generator=SEED)._cfg_dict(SEED, 0)
        h.sampler_init(cfgh, x0h, 1. / N_DIM**0.25, np.ones(N_DIM), x0h)
        h.sampler_run('HMC', 100, out_ptrs={})                         # step-size adaptation
        rh = h.sampler_run('HMC', 100, out_ptrs={})
        msh = h.last_kernel_ms()
        tfh = FLOPS_PER_LEAF * rh['total_tree_size'] / (msh * 1e-3) / 1e12
        hm[str(Ch)] = dict(chains_per_gpu=Ch, value=rh['total_tree_size'] / (msh * 1e-3), unit='leapfrog-steps*chains/s',
                           kernel='hmc_%s_kernel' % h.sampler_last_path(), kernel_ms=msh, roofline_frac=tfh / peak, achieved_tflops=tfh)
    extras['hmc_kernel'] = dict(n_int_step=32, iterations=100, outputs='none written (kernel only)', runs=hm,
                                note='hmc_team_kernel (8 chains per team of four warps) up to 4 groups per SM, hmc_dmma_kernel (8 chains per warp) above')
    # (b) the surrogate evaluation kernel alone: logp + gradient of 2^22 device-resident points
    Ce = 1 << 22
    Xe = torch.randn(Ce, N_DIM, dtype=torch.float64, device='cuda:%d' % dev) @ torch.tensor(np.linalg.cholesky(prob['cov']).T, device='cuda:%d' % dev)
    Xe = Xe.contiguous()
    lpe = torch.empty(Ce, dtype=torch.float64, device='cuda:%d' % dev)
    ge = torch.empty(Ce, N_DIM, dtype=torch.float64, device='cuda:%d' % dev)
    torch.cuda.synchronize(dev)
    mse = []
    for i in range(6):
        h.logp_and_grad_batch_dev(Xe.data_ptr(), Ce, lpe.data_ptr(), ge.data_ptr())
        mse.append(h.last_kernel_ms())
    mse = float(np.mean(mse[1:]))
    fe = (8 * N_DIM * N_DIM + 15 * N_DIM) * Ce
    extras['eval_kernel'] = dict(kernel='eval_dmma_kernel', points=Ce, ms=mse, points_per_s=Ce / mse * 1e3,
                                 algorithmic_flops_per_point=8 * N_DIM * N_DIM + 15 * N_DIM,
                                 roofline=dict(bound='tensor', achieved=fe / mse / 1e9, peak=peak, unit='TFLOP/s', frac=fe / mse / 1e9 / peak),
                                 hbm_gbs=Ce * (2 * N_DIM + 1) * 8 / mse / 1e6)
    del Xe, lpe, ge
    # (c) SURVEY 8f rank 1: the DES-Y1 example's three-module density (examples/des-y1-w-cosmosis.ipynb cells 9-18): n = 27 inputs with
    # module rescale + hard-bounded transform, m = 457 whitened outputs from a linear config and a quadratic config on the shared 9-D
    # mask, chi^2 likelihood, Gaussian prior on 13 inputs, radial bound -- fitted on the device, then batched logp + gradient and NUTS
    # on the tensor cores in feature form Phi(x) C^T (bfb_dmma.cuh, model variant bits 3|1|4).  Fractions are against the MINIMAL
    # algorithmic work 4 m P_f (P_f = 1 + 27 + 45 features), not against the n x n product per output the kernels used to do.
    try:
        pd_ = synthetic.des_y1_like(457)
        np_, mp_ = pd_['n'], pd_['m']
        surp = bfb.PolyModel([bfb.PolyConfig('linear'), bfb.PolyConfig('quadratic', input_mask=pd_['nonlinear'])], input_size=np_,
                             output_size=mp_, input_scales=pd_['ranges'], device=dev)
        denp = bfb.Density(surp, input_scales=pd_['ranges'], hard_bounds=True, likelihood=bfb.GaussianLikelihood(pd_['d'], np.ones(mp_), 0.),
                           prior=bfb.GaussianPrior(pd_['prior']['idx'], pd_['prior']['mu'], pd_['prior']['sig']))
        denp.fit(pd_['x_fit'], pd_['y_fit'])
        Pf = 1 + np_ + 45
        fl_min = 4 * mp_ * Pf
        hp = denp._sync(False)
        Cp = 1 << 16
        Xp = torch.tensor(denp.from_original(np.tile(pd_['x_0'], (Cp // pd_['x_0'].shape[0], 1))), device='cuda:%d' % dev).contiguous()
        lpp = torch.empty(Cp, dtype=torch.float64, device='cuda:%d' % dev)
        gp = torch.empty(Cp, np_, dtype=torch.float64, device='cuda:%d' % dev)
        torch.cuda.synchronize(dev)
        msp = []
        for i in range(5):
            hp.logp_and_grad_batch_dev(Xp.data_ptr(), Cp, lpp.data_ptr(), gp.data_ptr())
            msp.append(hp.last_kernel_ms())
        msp = float(np.mean(msp[1:]))
        ttp = bfb.sample(denp, dict(n_chain=C, n_iter=200, n_warmup=100, x_0=pd_['x_0'][:C], random_generator=SEED), verbose=False,
                         fields=('tree_depth',))
        extras['pipeline_kernel'] = dict(
            workload='des_y1_example_shape_n27_m457_shared_9d_mask_hard_bounds_prior_bound', features=Pf, algorithmic_flops_per_evaluation=fl_min,
            flops_note='minimal: 4 m P_f (value GEMM + gradient GEMM over the features); one n x n product per output would be m (2 n^2 + 5 n) = %d' % (mp_ * (2 * np_ * np_ + 5 * np_)),
            eval=dict(kernel={'lik_feat': 'likf_eval_dmma_kernel', 'lik_dmma': 'lik_eval_dmma_kernel'}.get(hp.eval_last_path(), hp.eval_last_path()),
                      points=Cp, ms=msp, points_per_s=Cp / msp * 1e3,
                      roofline=dict(bound='tensor', achieved=fl_min * Cp / msp / 1e9, peak=peak, unit='TFLOP/s', frac=fl_min * Cp / msp / 1e9 / peak)),
            nuts=dict(kernel='nuts_%s_kernel' % hp.sampler_last_path(), chains_per_gpu=C, iterations=200, kernel_ms=ttp.kernel_ms,
                      value=ttp.total_tree_size / ttp.kernel_ms * 1e3, unit='leapfrog-steps*chains/s',
                      roofline_frac=fl_min * ttp.total_tree_size / ttp.kernel_ms / 1e9 / peak, mean_tree_depth=float(ttp.arrays['tree_depth'].mean())))
        del Xp, lpp, gp, ttp
    except Exception as exc:                                   # supplementary measurement: never fails the bench line
        extras['pipeline_kernel'] = dict(error=repr(exc))

    # (d) the alternative NUTS kernel families on the headline run, kernel only (the one-warp-per-group kernel is the default: see
    # DESIGN.md 4.1): four-warp team per group (bfb_sampler_team.cu; HMC team is the default up to 4 groups per SM), and integrator
    # warp + tree warp per group with a speculative trajectory (bfb_sampler_pair.cu)
    for fam in ('team', 'pair'):
        try:
            os.environ['BFB200_SAMPLER'] = fam
            cfgt = bfb.NTrace(**trace_kw)._cfg_dict(SEED, 0)
            h.sampler_init(cfgt, x0, 1. / N_DIM**0.25, np.ones(N_DIM), x0)
            best = None
            for i in range(2):
                h.sampler_reset()
                flush.zero_()
                torch.cuda.synchronize(dev)
                rt = h.sampler_run('NUTS', N_ITER, out_ptrs={})
                mst = h.last_kernel_ms()
                if best is None or mst < best[1]:
                    best = (rt['total_tree_size'], mst)
            extras[fam + '_kernel'] = dict(kernel='nuts_%s_kernel' % h.sampler_last_path(), chains_per_gpu=C, value=best[0] / best[1] * 1e3,
                                           unit='leapfrog-steps*chains/s', kernel_ms=best[1],
                                           roofline_frac=FLOPS_PER_LEAF * best[0] / (best[1] * 1e-3) / 1e12 / peak)
        except Exception as exc:
            extras[fam + '_kernel'] = dict(error=repr(exc))
        finally:
            os.environ.pop('BFB200_SAMPLER', None)
    # (e) BASELINE configs[3]: 64-D cubic-3 stack (P = 47905), NUTS with per-chain divergent tree depths
    try:
        spec3, cov3 = synthetic.cubic3_stack(64, seed=3)
        h3 = _cabi.Handle(dev)
        h3.set_model(spec3)
        C3 = 1024
        x03 = (np.linalg.cholesky(cov3) @ np.random.default_rng(0).normal(size=(64, C3))).T
        cfg3 = bfb.NTrace(n_chain=C3, n_iter=300, n_warmup=100, x_0=x03, random_generator=SEED)._cfg_dict(SEED, 0)
        h3.sampler_init(cfg3, x03, 1. / 64**0.25, np.ones(64), x03)
        h3.sampler_run('NUTS', 100, out_ptrs={})
        r3 = h3.sampler_run('NUTS', 60, fields=('tree_depth',))
        ms3 = h3.last_kernel_ms()
        fam3 = h3.sampler_last_path()
        gen3 = None
        try:                                                     # the same 60 iterations on the generic warp-per-chain kernel
            os.environ['BFB200_SAMPLER'] = 'generic'
            h3.sampler_init(cfg3, x03, 1. / 64**0.25, np.ones(64), x03)
            h3.sampler_run('NUTS', 100, out_ptrs={})
            rg = h3.sampler_run('NUTS', 60, fields=('tree_depth',))
            gen3 = dict(kernel='nuts_%s_kernel' % h3.sampler_last_path(), kernel_ms=h3.last_kernel_ms(),
                        value=rg['total_tree_size'] / h3.last_kernel_ms() * 1e3)
        finally:
            os.environ.pop('BFB200_SAMPLER', None)
        fl3 = 8 * 64 * 64 + 24 * 64 + 1.5 * 64 * 63 * 62
        hist = np.bincount(r3['tree_depth'].ravel(), minlength=11)
        size = 2.**np.arange(len(hist))                      # leaves of a full tree of that depth
        extras['config3'] = dict(workload='64-D cubic-3 stack (P=47905), injected coefficients, 1024 chains', kernel='nuts_%s_kernel' % fam3,
                                 generic_kernel=gen3,
                                 iterations=60, kernel_ms=ms3, value=r3['total_tree_size'] / ms3 * 1e3, unit='leapfrog-steps*chains/s',
                                 algorithmic_flops_per_leapfrog=fl3, roofline_frac=fl3 * r3['total_tree_size'] / (ms3 * 1e-3) / 1e12 / peak,
                                 tree_depth_histogram=hist.tolist(), mean_tree_depth=float(r3['tree_depth'].mean()),
                                 lockstep_efficiency=float((hist * size).sum() / (hist.sum() * size[np.nonzero(hist)[0].max()])),
                                 note='lockstep_efficiency: mean tree size over the size of the deepest tree = the row utilisation a kernel '
                                      'keeping all chains in lock step per iteration would have; the kernels here let every chain run on')
        h3.close()
    except Exception as exc:
        extras['config3'] = dict(error=repr(exc))
    # (g) tempered NUTS (TNUTS, SURVEY 8f rank 4): the headline target + a quadratic base density, warp-per-chain kernel
    try:
        sb = bfb.PolyModel('quadratic', input_size=N_DIM, output_size=1)
        sb.fit(prob['x_fit'] * 1.5, prob['y_fit'] / 3., logp=prob['y_fit'][:, 0] / 3.)
        base = bfb.Density(sb)
        ttn = None
        for i in range(2):
            ttn = bfb.sample(den, bfb.TNTrace(base, 0., n_chain=C, n_iter=200, n_warmup=100, x_0=x0, random_generator=SEED,
                                              u_0=np.zeros(C)), verbose=False, fields=('tree_size', 'weight'))
        extras['tempered_kernel'] = dict(kernel='tsampler_kernel (one warp per chain)', sampler='TNUTS', chains_per_gpu=C, iterations=200,
                                         kernel_ms=ttn.kernel_ms, value=ttn.total_tree_size / ttn.kernel_ms * 1e3,
                                         unit='leapfrog-steps*chains/s', density_evaluations_per_leapfrog=4,
                                         evaluations_per_s=4 * ttn.total_tree_size / ttn.kernel_ms * 1e3,
                                         mean_tree_size=float(ttn.arrays['tree_size'].mean()))
        del ttn
    except Exception as exc:
        extras['tempered_kernel'] = dict(error=repr(exc))
    # (f) e2e variants through the public API (one timed call each after a warm call)
    try:
        ev = {}
        for name, kw in (('all_records', dict(keep='all')), ('post_warmup_thin10_summaries', dict(keep='post_warmup', thin=10, summaries=True))):
            tt = None
            for i in range(2):
                del tt                                   # hand the pinned output buffers back to the pool before the next call
                flush.zero_()
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                tt = bfb.sample(den, dict(trace_kw), verbose=False, **kw)
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
            ev[name] = dict(value=tt.total_tree_size / dt, ms_per_step=dt * 1e3, kernel_ms=tt.kernel_ms,
                            d2h_bytes_per_step=int(sum(v.nbytes for k, v in tt.arrays.items() if k not in ('samples_original', 'logp_original'))))
            del tt
        extras['e2e_variants'] = ev
    except Exception as exc:
        extras['e2e_variants'] = dict(error=repr(exc))
    return extras


def fit_sweep(torch, dist, dev, rank, world, peak_dmma=None):
    """BASELINE configs[4]: cubic-2 fit, d = 32 (P = 1585), N = 1e4 .. 1e7 rows resident on the device(s): Gram kernel time
    (CUDA events) and algorithmic TFLOP/s = N P (P + 1) / t; with world > 1 the rows are sharded and the packed exchange
    buffer is all-reduced over NCCL (timed), then every rank solves."""
    import ctypes as CT
    import bayesfast_b200 as bfb
    from bayesfast_b200 import _cabi
    from bayesfast_b200.fit import _allreduce_buffer
    n = 32
    sur = bfb.PolyModel('cubic-2', input_size=n, output_size=1, device=dev)
    P = sur.n_param
    h = sur._dev()
    h.set_model(sur.to_spec(with_bound=False))
    L = _cabi.lib()
    peak = peak_dmma or h.fp64_peak(1)
    d = torch.device('cuda', dev)
    rows = []
    for N in (10**4, 10**5, 10**6, 10**7):
        Nl = N // world
        g = torch.Generator(device=d).manual_seed(1000 + rank)
        x = torch.randn(Nl, n, dtype=torch.float64, device=d, generator=g)
        coef = torch.randn(n, dtype=torch.float64, device=d, generator=torch.Generator(device=d).manual_seed(7))
        y = (-0.5 * (x * x).sum(1) + x @ coef + 0.05 * (x ** 3).sum(1)
             + 1e-3 * torch.randn(Nl, dtype=torch.float64, device=d, generator=g))[:, None].contiguous()
        torch.cuda.synchronize(d)
        best, ex = 1e30, {}
        for rep in range(3 if N < 10**7 else 2):
            _cabi.check(L.bfb_fit_begin(h._h, None))
            _cabi.check(L.bfb_fit_accumulate(h._h, x.data_ptr(), y.data_ptr(), None, Nl, _cabi.BFB_DEVICE))
            best = min(best, h.last_kernel_ms())
            if world > 1:
                dist.barrier()
                st = {}
                _allreduce_buffer(h, None, st)
                if not ex or st['allreduce_s'] < ex['allreduce_s']:
                    ex = st
        t0 = time.time()
        out = np.empty(P)
        rr = CT.c_double(0)
        _cabi.check(L.bfb_fit_solve(h._h, out.ctypes.data_as(_cabi._dp), CT.byref(rr)))
        solve_s = time.time() - t0
        if world > 1:
            t = torch.tensor([best], dtype=torch.float64, device=d)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            best = float(t[0])
        flops = float(Nl * world) * P * (P + 1) + 2. * Nl * world * P
        row = dict(N=Nl * world, rows_per_gpu=Nl, P=P, gram_ms=best, tflops_all_gpus=flops / (best * 1e-3) / 1e12,
                   frac_of_fp64_peak=flops / (best * 1e-3) / 1e12 / (peak * world), solve_s=solve_s, rel_resid=rr.value)
        if ex:
            row.update(allreduce_ms=ex['allreduce_s'] * 1e3, allreduce_bytes=ex['allreduce_bytes'],
                       allreduce_gbs=ex['allreduce_bytes'] / ex['allreduce_s'] / 1e9)
        rows.append(row)
        del x, y
    return dict(workload='PolyModel cubic-2 fit sweep, d=32, P=1585, rows resident on the device(s)', n_gpus=world, fp64_peak_tflops_per_gpu=peak,
                rows=rows)


def dump_outputs(out_dir, d_out, total_tree_size, C, max_bytes=64 * 10**6, seed=0):
    """Writes what the last timed step handed back: every output array of sampler_run, laid out [chain, iteration(, dim)],
    for a seeded sample of whole chains (all 4096 chains are 1.8 GB; the sample fits max_bytes), plus its total_tree_size.
    Integer statistics are stored as float64 (exact).  The inputs and the chain sample depend only on the arguments, so two
    builds run with the same arguments can be compared file by file.  Called on rank 0 only: with several GPUs the files
    cover rank 0's C chains (and their total_tree_size), not the other ranks' share of the step."""
    import torch
    bytes_per_chain = 8 * N_ITER * (N_DIM + len(d_out) - 1)         # float64 samples + one float64 per statistic
    n_keep = min(C, (max_bytes - 4096) // bytes_per_chain)           # 4096: the .npy headers
    chains = np.sort(np.random.default_rng(seed).choice(C, size=n_keep, replace=False))
    idx = torch.from_numpy(chains).to(d_out['samples'].device)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in d_out.items():
        a = v.view(C, N_ITER, N_DIM) if k == 'samples' else v.view(C, N_ITER)
        np.save(os.path.join(out_dir, k + '.npy'), a.index_select(0, idx).to(torch.float64).cpu().numpy())
    np.save(os.path.join(out_dir, 'total_tree_size.npy'), np.array(float(total_tree_size)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5, help='timed steps (at least 1)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy; with several GPUs only rank 0 '
                         'writes, covering its own chains (see dump_outputs)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--chains-per-gpu', type=int, default=CHAINS_PER_GPU)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-budget', type=float, default=15.)
    ap.add_argument('--no-extras', action='store_true', help='skip the more_chains / eval_kernel supplementary measurements')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 implementation')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))

    from bayesfast_b200 import synthetic
    C = args.chains_per_gpu
    prob = synthetic.des_shaped(N_DIM, seed=1, n_chain=C * max(world, 1), order=ORDER)
    config = dict(workload=WORKLOAD, n=N_DIM, order=ORDER, n_param=synthetic.n_param(ORDER, N_DIM),
                  chains_per_gpu=C, n_iter=N_ITER, n_warmup=N_WARMUP, n_fit=int(prob['x_fit'].shape[0]),
                  step='one full NUTS run of all chains (one kernel launch)',
                  l2='256 MiB scratch memset between timed steps (L2 flush); outputs (1.8 GB/step) exceed L2',
                  parallelism='chains sharded over {} GPU(s), no data-path collective'.format(world))

    if args.impl == 'reference':
        if rank != 0:
            return
        cores = cpu_cores()
        vals, cb = [], None
        for s_ in range(args.warmup + args.steps):
            cb = run_reference_python(prob, cores, per=1)
            if cb is None or 'error' in cb:
                break
            if s_ >= args.warmup:
                vals.append((cb['leaves'], cb['seconds']))
        if cb is None or 'error' in cb:             # not installed on this box: the C port of the same path
            why = 'baseline/_ref missing' if cb is None else cb['error']
            spec = oracle_spec_cpu(prob)
            vals = []
            for s_ in range(args.warmup + args.steps):
                cb, leaves, dt = run_cpu_baseline(spec, prob, budget_s=min(args.cpu_budget, 10.))
                if s_ >= args.warmup:
                    vals.append((leaves, dt))
            cb['fallback'] = why
        leaves = sum(v[0] for v in vals)
        dt = sum(v[1] for v in vals)
        cb['value'] = leaves / dt
        print(json.dumps(dict(metric='nuts_leapfrog_steps_x_chains_per_s', value=leaves / dt, unit='leapfrog-steps*chains/s',
                              impl='reference', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                              ms_per_step=dt / max(args.steps, 1) * 1e3, higher_is_better=True, scaling='weak',
                              vs_baseline=None, dtype='f64', data='synthetic', config=config, cpu_baseline=cb,
                              e2e=dict(value=leaves / dt, unit='leapfrog-steps*chains/s', h2d_bytes_per_step=0,
                                       d2h_bytes_per_step=0), gpu_launches=0)))
        return

    import torch
    import torch.distributed as dist
    import bayesfast_b200 as bfb
    from bayesfast_b200 import _cabi
    numa_cpus = None
    if world > 1:
        from bayesfast_b200.runtime import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local)       # host buffers of this rank on the NUMA node of its GPU
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = local

    # ---- setup (untimed): fit the surrogate on the GPU, build the density ----
    sur = bfb.PolyModel(ORDER, input_size=N_DIM, output_size=1, device=dev)
    t0 = time.time()
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    fit_s = time.time() - t0            # first call of the process: CUDA context, module load and allocations included
    t0 = time.time()
    sur.fit(prob['x_fit'], prob['y_fit'], logp=prob['y_fit'][:, 0])
    fit_warm_s = time.time() - t0       # the same fit again (steady state: host copies, Gram kernel, solve, bound)
    den = bfb.Density(sur)
    h = den._sync(False)
    peak = max(h.fp64_peak(0) for _ in range(2))               # TFLOP/s, DFMA, measured now on this GPU
    x0 = np.ascontiguousarray(prob['x_0'][rank * C:(rank + 1) * C])
    trace_kw = dict(n_chain=C, n_iter=N_ITER, n_warmup=N_WARMUP, x_0=x0, random_generator=SEED)
    cfg = bfb.NTrace(**trace_kw)._cfg_dict(SEED, rank * C)
    h.sampler_init(cfg, x0, 1. / N_DIM**0.25, np.ones(N_DIM), x0)
    S = C * N_ITER
    d_out = dict(samples=torch.empty(S * N_DIM, dtype=torch.float64, device='cuda:%d' % dev))
    for k in _cabi.FLOAT_STATS:
        d_out[k] = torch.empty(S, dtype=torch.float64, device='cuda:%d' % dev)
    for k in _cabi.INT_STATS:
        d_out[k] = torch.empty(S, dtype=torch.int32, device='cuda:%d' % dev)
    ptrs = {k: v.data_ptr() for k, v in d_out.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:%d' % dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        h.synchronize()

    def one_step():
        h.sampler_reset()
        r = h.sampler_run('NUTS', N_ITER, out_ptrs=ptrs)
        return r['total_tree_size'], h.last_kernel_ms()

    for _ in range(args.warmup):
        one_step()
        flush.zero_()
    barrier()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, dev), daemon=True)
    th.start()
    l0 = h.launch_count()
    leaves = 0
    kern_ms = []
    step_ms = 0.
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        lv, kms = one_step()                  # returns after the stream has been synchronised
        barrier()
        step_ms += (time.perf_counter() - t0) * 1e3
        leaves += lv
        kern_ms.append(kms)
    launches = h.launch_count() - l0
    kernel_family = h.sampler_last_path()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out, lv, C)
    # device time of the timed steps: CUDA events around the kernel on the launching stream (+ the reset copies,
    # which the wall clock above includes); report the event time, max over ranks
    dev_ms = float(sum(kern_ms))
    if world > 1:
        t = torch.tensor([dev_ms, step_ms], dtype=torch.float64, device='cuda:%d' % dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, step_ms = float(t[0]), float(t[1])
        t = torch.tensor([leaves, launches], dtype=torch.int64, device='cuda:%d' % dev)
        dist.all_reduce(t)
        leaves_all, launches_all = int(t[0]), int(t[1])
    else:
        leaves_all, launches_all = leaves, launches
    value = leaves_all / (step_ms * 1e-3)

    # ---- e2e: the public API, host buffers in and out ----
    e2e_leaves, e2e_ms, h2d, d2h, e2e_kernel_ms = 0, 0., 0, 0, 0.
    n_e2e = max(1, min(args.steps, 3))
    for i in range(1 + n_e2e):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        tt = bfb.sample(den, dict(trace_kw), verbose=False, keep='post_warmup')
        barrier()
        if i > 0:
            e2e_ms += (time.perf_counter() - t0) * 1e3
            e2e_kernel_ms += tt.kernel_ms
            e2e_leaves += tt.total_tree_size
            h2d = x0.nbytes * 2 + 8 * C + x0.nbytes
            d2h = sum(v.nbytes for k, v in tt.arrays.items() if k not in ('samples_original', 'logp_original'))
            # step_size / step_size_bar are constant per chain after the warm-up: one column of each crosses PCIe, the host
            # replicates it (bfb_sampler.cu: single_launch_host_outputs)
            d2h -= sum(tt.arrays[k].nbytes - 8 * C for k in ('step_size', 'step_size_bar') if k in tt.arrays)
        del tt
    stop.set()
    th.join(timeout=2)
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device='cuda:%d' % dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t[0])
        t = torch.tensor([e2e_leaves], dtype=torch.int64, device='cuda:%d' % dev)
        dist.all_reduce(t)
        e2e_leaves = int(t[0])
    e2e_value = e2e_leaves / (e2e_ms * 1e-3)

    fsweep = None
    if not args.no_extras:
        try:
            fsweep = fit_sweep(torch, dist, dev, rank, world)        # all ranks: rows sharded, the exchange buffer all-reduced over NCCL
        except Exception as exc:
            fsweep = dict(error=repr(exc))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    k_ms = float(np.mean(kern_ms))
    achieved = FLOPS_PER_LEAF * (leaves / args.steps) / (k_ms * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get('sampler_kernel_dram_bytes_per_launch')
    except Exception:
        pass
    hbm_bytes = (leaves / args.steps) * 0 + C * N_ITER * (N_DIM * 8 + 7 * 8 + 3 * 4)
    roofline = dict(bound='tensor', pipe='FP64 pipe: the kernel evaluates the surrogate with m8n8k4 DMMAs; DFMA and DMMA issue to the same '
                    'pipe (measured 37.0 vs 37.2 TFLOP/s, 31 when interleaved)', kernel='nuts_%s_kernel' % kernel_family, achieved=achieved, peak=peak, unit='TFLOP/s',
                    frac=achieved / peak, traffic=traffic,
                    peak_source='bfb_fp64_peak DFMA microbenchmark run just before the timed region on this GPU '
                                '(MEASURED_PEAKS.json has no FP64 entry; nominal 37 TFLOP/s)',
                    algorithmic_flops_per_leapfrog=FLOPS_PER_LEAF, kernel_ms=k_ms,
                    hbm=dict(algorithmic_bytes_per_launch=hbm_bytes, achieved_gbs=hbm_bytes / (k_ms * 1e-3) / 1e9,
                             peak_gbs=peaks.get('hbm_gbs'), note='outputs only; the tree state stays in shared memory'))
    extras = {}
    if fsweep is not None:
        extras['fit_sweep'] = fsweep
    if not args.no_extras and world == 1:
        extras.update(extra_measurements(args, bfb, torch, den, h, prob, x0, trace_kw, flush, peak, dev, C))
    out = dict(metric='nuts_leapfrog_steps_x_chains_per_s', value=value, unit='leapfrog-steps*chains/s', n_gpus=world,
               steps=args.steps, warmup=args.warmup, ms_per_step=step_ms / args.steps, higher_is_better=True,
               scaling='weak', vs_baseline=None, dtype='f64', data='synthetic', config=config,
               e2e=dict(value=e2e_value, unit='leapfrog-steps*chains/s', h2d_bytes_per_step=int(h2d),
                        d2h_bytes_per_step=int(d2h), ms_per_step=e2e_ms / n_e2e, kernel_ms_per_step=e2e_kernel_ms / n_e2e,
                        api="bayesfast_b200.sample(density, trace, keep='post_warmup'): samples + 10 statistics of the {} post-warm-up "
                            "iterations of every chain to pinned host memory (one launch for the warm-up, one for the kept iterations "
                            "whose finished chunks are copied out while it runs; the two per-chain constant step-size statistics cross PCIe as one "
                            "column each and are replicated by the host thread)".format(N_ITER - N_WARMUP),
                        numa_cpus_rank0=(len(numa_cpus) if numa_cpus else None)),
               gpu_launches=int(launches_all), roofline=roofline, clocks=summarize_clocks(samples),
               fit=dict(seconds=fit_s, seconds_warm=fit_warm_s, kernel_ms=getattr(sur, '_fit_kernel_ms', None), n=N_DIM,
                        P=config['n_param'], N=config['n_fit'], rel_resid=getattr(sur, '_fit_rel_resid', None)),
               mean_tree_size=leaves / args.steps / (C * N_ITER), kernel='nuts_%s_kernel' % kernel_family, **extras)
    if world == 1 and not args.no_cpu_baseline:
        cores = cpu_cores()
        port = run_cpu_baseline(den.to_spec(), prob, budget_s=args.cpu_budget)[0]
        ref = run_reference_python(prob, cores, per=2)
        if ref is not None and 'error' not in ref:
            out['cpu_baseline'] = dict(ref, port=port)
        else:
            out['cpu_baseline'] = dict(port, reference=ref)
        out['cpu_baseline']['note'] = ('absolute rates with their core counts; the GPU/CPU ratio depends on how many cores the box has '
                                       '(round 1: 16 and 32 cores gave ratios 82 and 45 for the same GPU number)')
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
