"""Static SASS size of one kernel per named section of its source file.

usage: sass_sections.py OBJ KERNEL SOURCE [--group NAME=SEC+SEC+...] [--local]

OBJ is an object file, shared library or cubin holding sm_100a code built with -lineinfo; KERNEL is a substring of the kernel's
mangled name (e.g. nuts_dmma_kernelILi7ELi1ELi4E); SOURCE is the .cu file that defines it.  Sections start at marker comments
`// section: <name>` in SOURCE and run to the next marker.  Every instruction is attributed to its outermost source location
(nvdisasm --print-line-info-inline): code inlined from headers counts where the kernel calls it, out-of-line subroutines
(__noinline__ functions placed in the kernel's text) count under the file that defines them.  --group prints the sum of
several sections; --local lists the local-memory instructions (spills, indexed arrays) with their source lines.

example (the per-round code of the headline NUTS kernel):
  make -C bayesfast_b200/csrc bfb_sampler_dmma_headline.o
  python scripts/sass_sections.py bayesfast_b200/csrc/bfb_sampler_dmma_headline.o nuts_dmma_kernelILi7ELi1ELi4E \\
      bayesfast_b200/csrc/bfb_sampler_dmma.cu --group tree=leaf+merge+push+extend \\
      --group round='round start+evaluation+leaf+merge+push+extend'
"""
import argparse
import bisect
import collections
import glob
import os
import re
import subprocess
import sys
import tempfile

INSN = re.compile(r'\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)')
LOC = re.compile(r'"([^"]+)", line (\d+)')
MARK = re.compile(r'//\s*section:\s*(.+?)\s*$')


def cubins(path, tmp):
    if path.endswith('.cubin'):
        return [path]
    subprocess.run(['cuobjdump', '-xelf', 'all', os.path.abspath(path)], cwd=tmp, check=True, capture_output=True)
    return sorted(glob.glob(os.path.join(tmp, '*.cubin')))


def kernel_text(path, kernel):
    """(mangled name, disassembly lines of its .text section) of the first kernel whose name contains `kernel`."""
    with tempfile.TemporaryDirectory() as tmp:
        for cb in cubins(path, tmp):
            txt = subprocess.run(['nvdisasm', '--print-line-info-inline', cb], check=True, capture_output=True,
                                 text=True).stdout
            name, body = None, []
            for ln in txt.splitlines():
                m = re.match(r'\s*\.section\s+\.text\.(\S+?),', ln)
                if m:
                    if name:
                        return name, body
                    name = m.group(1) if kernel in m.group(1) else None
                    continue
                if name:
                    body.append(ln)
            if name:
                return name, body
    sys.exit('no kernel matching %r in %s' % (kernel, path))


def markers(source):
    lines, names = [], []
    with open(source) as f:
        for i, ln in enumerate(f, 1):
            m = MARK.search(ln)
            if m:
                lines.append(i)
                names.append(m.group(1))
    if not lines:
        sys.exit('no "// section: <name>" markers in ' + source)
    return lines, names


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('obj')
    ap.add_argument('kernel')
    ap.add_argument('source')
    ap.add_argument('--group', action='append', default=[], metavar='NAME=SEC+SEC')
    ap.add_argument('--local', action='store_true')
    a = ap.parse_args()
    mlines, mnames = markers(a.source)
    src = os.path.basename(a.source)
    name, body = kernel_text(a.obj, a.kernel)

    def section(loc):
        if loc is None:
            return '(no line info)'
        f, line = loc
        if os.path.basename(f) != src:
            return 'out of line: ' + os.path.basename(f)
        i = bisect.bisect_right(mlines, line) - 1
        return mnames[i] if i >= 0 else '(before the first marker)'

    count, local = collections.Counter(), []
    loc = None
    for ln in body:
        if ln.lstrip().startswith('//##'):
            found = LOC.findall(ln)
            loc = (found[-1][0], int(found[-1][1])) if found else None
            continue
        m = INSN.match(ln)
        if m:
            count[section(loc)] += 1
            if a.local and m.group(1).split('.')[0] in ('LDL', 'STL'):
                local.append((m.group(1), loc))
    total = sum(count.values())
    print(name)
    print('%-34s %7s %9s' % ('section', 'insns', 'KB'))
    order = [n for n in mnames if n in count] + sorted(k for k in count if k not in mnames)
    for k in order:
        print('%-34s %7d %9.1f' % (k, count[k], count[k] * 16 / 1024))
    print('%-34s %7d %9.1f' % ('total', total, total * 16 / 1024))
    for g in a.group:
        gname, secs = g.split('=', 1)
        secs = secs.split('+')
        unknown = [s for s in secs if s not in mnames]
        if unknown:
            sys.exit('unknown section(s) in --group %s: %s' % (gname, ', '.join(unknown)))
        n = sum(count[s] for s in secs)
        print('group %-28s %7d %9.1f   (%s)' % (gname, n, n * 16 / 1024, ' + '.join(secs)))
    for op, l in local:
        print('local memory: %-10s %s' % (op, '%s:%d' % (os.path.basename(l[0]), l[1]) if l else '(no line info)'))


if __name__ == '__main__':
    main()
