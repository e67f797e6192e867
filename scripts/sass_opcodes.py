"""Static SASS opcode histogram of the main kernels of libbfb200 (cuobjdump -sass of the in-tree objects; no GPU needed).
usage: python scripts/sass_opcodes.py > profiles/rNN_sass_opcodes.md"""
import collections, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CS = os.path.join(ROOT, 'bayesfast_b200', 'csrc')
KERNELS = [('bfb_sampler_dmma_headline.o', 'nuts_dmma_kernelILi7ELi1ELi4E', 'nuts_dmma_kernel<7,1,4> (headline: d=26 cubic-2 NUTS, 8 chains per warp)'),
           ('bfb_sampler_dmma_headline.o', 'hmc_dmma_kernelILi7ELi1ELi8E', 'hmc_dmma_kernel<7,1,8>'),
           ('bfb_sampler_team.o', 'nuts_team_kernelILi16ELi5EE', 'nuts_team_kernel<16,5> (64-D cubic-3, 8 chains per team of four warps)'),
           ('bfb_sampler_team.o', 'hmc_team_kernelILi7ELi1ELi4E', 'hmc_team_kernel<7,1,4>'),
           ('bfb_sampler_pair.o', 'nuts_pair_kernelILi7ELi1ELi4E', 'nuts_pair_kernel<7,1,4> (integrator warp + tree warp per 8-chain group)'),
           ('bfb_sampler_dmma.o', 'nuts_dmma_kernelILi7ELi10ELi4E', 'nuts_dmma_kernel<7,10,4> (DES-shaped likelihood pipeline: bound + rescale + transform + prior)'),
           ('bfb_eval_dmma.o', 'eval_dmma_kernelILi7ELi1E', 'eval_dmma_kernel<7,1> (batched logp + gradient)'),
           ('bfb_lik_dmma.o', 'lik_eval_dmma_kernelILi7ELi2ELb1E', 'lik_eval_dmma_kernel<7,2,true>'),
           ('bfb_fit.o', 'gram_kernel', 'gram_kernel (fit: fused feature expansion + DMMA Gram)'),
           ('bfb_post.o', 'bitonic_shared_kernel', 'bitonic_shared_kernel (SystematicResampler argsort)')]
print('# SASS opcode histograms (static, `cuobjdump -sass`, sm_100a) of the main kernels\n')
print('FP64 tensor path = `DMMA` (`mma.sync.aligned.m8n8k4.f64`; tcgen05 has no FP64 kind, so no `UTC*MMA`), staging with `LDGSTS` '
      '(`cp.async`) where an operand is streamed; no `UTMALDG` (records of 7.5 KB per output / 28 KB tables staged once do not need TMA).\n')
for obj, pat, title in KERNELS:
    txt = subprocess.run(['cuobjdump', '-sass', os.path.join(CS, obj)], capture_output=True, text=True).stdout
    ops = collections.Counter(); active = False; name = None
    for ln in txt.splitlines():
        m = re.search(r'Function : (\S+)', ln)
        if m:
            active = pat in m.group(1) and name in (None, m.group(1))
            if active: name = m.group(1)
            continue
        if not active: continue
        m = re.match(r'\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)', ln)
        if m: ops[m.group(1)] += 1
    tot = sum(ops.values())
    if not tot:
        print('## %s\n\nnot found in %s\n' % (title, obj)); continue
    print('## %s\n\n%d instructions (%d KB).  ' % (title, tot, tot * 16 // 1024) + ', '.join('`%s` %d' % kv for kv in ops.most_common(18)) + '\n')
    keys = ('DMMA', 'DFMA', 'DADD', 'DMUL', 'LDGSTS', 'LDS', 'STS', 'LDG', 'STG', 'SHFL', 'BAR', 'HMMA', 'UTCHMMA', 'UTMALDG')
    print('| ' + ' | '.join(keys) + ' |\n|' + '---|' * len(keys) + '\n| ' + ' | '.join(str(ops.get(k, 0)) for k in keys) + ' |\n')
