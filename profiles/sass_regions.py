"""Static SASS instruction counts of one kernel, per source region (CPU only: cuobjdump + nvdisasm from the CUDA toolkit).

    python profiles/sass_regions.py nnest_b200/lib/obj/nnb_tc_d30.o [kernel-substring] [--csrc DIR]

The kernel defaults to mcmc_tc_kernel<0,1,30> (the c4 step kernel).  Every instruction is attributed, through the inlining
chain that `nvdisasm -gi` prints (needs a -lineinfo build, as nnest_b200/build.py does), to the innermost source location
that falls into one of the regions below; the rest is "other".  Regions are found in the sources by function name or by
marker lines (a marker that a source does not have is skipped), so the script keeps working when line numbers move;
--csrc names the sources the object was built from (default: the tree's nnest_b200/csrc).  Counts are static
(instructions in the binary), not executed instructions.
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'nnest_b200', 'csrc')
# (name, file, how): ('fn', function-name regex) spans the function's body; ('mark', start regex, end regex) spans the lines from
# the first match of start to the next match of end.  Regions of one file must not overlap.
REGIONS = [
    ('split_tf32', 'nnb_tc.cuh', ('fn', 'split_tf32')),
    ('tmem_st (callers own them)', 'nnb_tc.cuh', ('mark', r'void tmem_st8\(', r'^// hi = x truncated')),
    ('tanh', 'nnb_tc_kernels.cuh', ('fn', 'tc_tanh_scaled2?')),
    ('hidden epilogue', 'nnb_tc_kernels.cuh', ('fn', 'tc_hidden_epilogue')),
    ('layer-1 input (first block)', 'nnb_tc_kernels.cuh', ('mark', r'---- layer 1: A = masked inputs', r'const uint32_t b_hi = wsm_u32')),
    ('output epilogue', 'nnb_tc_kernels.cuh', ('mark', r'x = \(z - t\) \* exp\(-log_s\)', r'if \(k == 0\) ld \*=')),
    ('output epilogue', 'nnb_tc_kernels.cuh', ('mark', r'^// Output epilogue of a coupling block', r'^// Flow inverse of one tile')),
    ('rosenbrock (inline)', 'nnb_tc_kernels.cuh', ('mark', r'the config-4 target inline', r'lp = isfinite\(out\)')),
    ('box_muller', 'nnb_device.cuh', ('fn', 'box_muller4?')),
    ('philox', 'nnb_device.cuh', ('fn', 'philox4x32_10')),
]
OPS = ['FADD', 'FADD2', 'FMUL', 'FMUL2', 'FFMA', 'FFMA2', 'FSETP', 'FMNMX', 'LOP3', 'MUFU', 'MOV', 'PRMT', 'STTM', 'LDTM',
       'R2UR', 'STS', 'LDS']


def fn_span(lines, name):
    """1-based (first, last) lines of every definition of a function whose name matches `name` (overloads included)."""
    spans = []
    for i, l in enumerate(lines):
        if re.match(r'\s*(static\s+)?__device__\b.*\b(%s)\s*\(' % name, l):
            depth, seen = 0, False
            for j in range(i, len(lines)):
                depth += lines[j].count('{') - lines[j].count('}')
                seen = seen or '{' in lines[j]
                if seen and depth == 0:
                    spans.append((i + 1, j + 1))
                    break
    return spans


def region_spans(csrc):
    out = []
    for name, fname, how in REGIONS:
        lines = open(os.path.join(csrc, fname)).read().split('\n')
        if how[0] == 'fn':
            spans = fn_span(lines, how[1])
            assert spans, (name, how)
        else:
            a = next((i for i, l in enumerate(lines) if re.search(how[1], l)), None)
            if a is None:
                continue
            b = next(i for i in range(a + 1, len(lines)) if re.search(how[2], lines[i]))
            spans = [(a + 1, b + 1)]
        out += [(name, fname, s) for s in spans]
    return out


def classify(chain, spans):
    for fname, line in chain:            # innermost first
        for name, f, (a, b) in spans:
            if f == fname and a <= line <= b:
                return name
    return 'other'


def main():
    args = sys.argv[1:]
    csrc = CSRC
    if '--csrc' in args:
        k = args.index('--csrc')
        csrc = args[k + 1]
        del args[k:k + 2]
    obj = args[0]
    want = args[1] if len(args) > 1 else 'mcmc_tc_kernelILi0ELi1ELi30E'
    spans = region_spans(csrc)
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(['cuobjdump', '-xelf', 'all', os.path.abspath(obj)], cwd=tmp, check=True, capture_output=True)
        cubins = [f for f in os.listdir(tmp) if f.endswith('.cubin')]
        assert len(cubins) == 1, cubins
        sass = subprocess.run(['nvdisasm', '-gi', '-c', os.path.join(tmp, cubins[0])], check=True, capture_output=True,
                              text=True).stdout
    fn, chain, fresh = None, [], False
    counts = collections.defaultdict(collections.Counter)
    for l in sass.split('\n'):
        m = re.match(r'^\.text\.(\S+):', l)
        if m:
            fn = m.group(1)
            continue
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', l)
        if m:
            if not fresh:
                chain = []
            fresh = True
            chain.append((os.path.basename(m.group(1)), int(m.group(2))))
            continue
        m = re.match(r'\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)(\.\S+)?', l)
        if m:
            fresh = False
            if fn is None or want not in fn:
                continue
            op = m.group(1)
            if op in ('IMAD', 'UMOV') and m.group(2) and m.group(2).startswith('.MOV'):
                op = 'MOV'
            region = classify(chain, spans)
            counts[region][op] += 1
            counts[region]['total'] += 1
            counts['(kernel)'][op] += 1
            counts['(kernel)']['total'] += 1
    assert counts, 'no kernel matching %r in %s' % (want, obj)
    names = [n for n, _, _ in spans]
    order = sorted(set(names), key=names.index) + ['other', '(kernel)']
    cols = OPS + ['total']
    print('kernel: %s' % want)
    print('%-28s' % 'region' + ''.join('%7s' % c for c in cols))
    for r in order:
        if r in counts:
            print('%-28s' % r + ''.join('%7d' % counts[r][c] for c in cols))


if __name__ == '__main__':
    main()
