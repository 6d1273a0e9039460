"""FP64 operations per processed cell of every kernel class, counted in the SASS of the built library (DFMA = 2 flop, DMUL/DADD = 1;
MUFU-based reciprocal / square-root / log sequences are expanded into those by the compiler and so are included).  Straight-line
kernels: whole body, which includes rarely taken slow paths -> an upper bound; k_step: the two sweep loops (per interval).
Writes profiles/fp64_ops.json, which bench.py reads for the FP64 view of the roofline."""
import collections, json, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = os.path.join(ROOT, 'ms-eetc_b200', 'mseetc', 'libmseetc_b200.so')
sass = subprocess.run(['cuobjdump', '-sass', lib], capture_output=True, text=True).stdout
funcs, cur = {}, None
for line in sass.splitlines():
    m = re.search(r'Function : (\S+)', line)
    if m:
        cur = m.group(1); funcs[cur] = []; continue
    m = re.match(r'\s+/\*([0-9a-f]{4,})\*/\s+(.*?);', line)
    if m and cur:
        funcs[cur].append((int(m.group(1), 16), re.sub(r'^@!?U?P\d\s+', '', m.group(2).strip())))


def flops(ins):
    c = collections.Counter(t.split()[0].split('.')[0] for _, t in ins)
    return 2 * c['DFMA'] + c['DMUL'] + c['DADD'], sum(c.values())


def find(sub):
    return [k for k in funcs if sub in k]


out = {}
# 'cell_trial' = evaluation at the trial point (k_cell_trial_eval: the kernel of every iteration), 'cell_eval' = the same at the
# starting point (once per solve)
for cls, sub in (('cell_trial', 'k_cell_trial_evalE'), ('cell_eval', 'k_cell_evalE'), ('cell_step', 'k_cell_stepE'),
                 ('cell_trial_dyn', 'k_cell_trial_eval_dynE'), ('cell_eval_dyn', 'k_cell_eval_dynE')):
    f, n = flops(funcs[find(sub)[0]])
    out[cls] = {'flop_per_cell': f, 'instructions': n}
ks = funcs[[k for k in find('k_stepILi32ELi8EE')][0]]
loops = []
for a, t in ks:
    m = re.search(r'BRA\s+(?:U?P\d,\s*)?(0x[0-9a-f]+)', t)
    if m and int(m.group(1), 16) < a:
        loops.append((int(m.group(1), 16), a))
def body(lo, hi):
    return [i for i in ks if lo <= i[0] <= hi]


def n_ldgsts(lo, hi):
    return sum(1 for _, t in body(lo, hi) if t.startswith('LDGSTS'))


# the sweep loops are recognised by their prefetch instructions: 23 fields backward (plain variant = the shorter one), 14 forward
bwd = min((l for l in loops if n_ldgsts(*l) == 23), key=lambda l: l[1] - l[0])
fwd = min((l for l in loops if n_ldgsts(*l) == 14), key=lambda l: l[1] - l[0])
f = n = 0
for lo, hi in (bwd, fwd):
    a, b = flops(body(lo, hi)); f += a; n += b
out['inst_step_sequential'] = {'flop_per_cell': f, 'instructions': n, 'note': 'k_step: backward (plain variant) + forward loop body per interval'}
# parallel-in-time sweeps: element pass + in-chunk recursion + forward sweep per interval (loop bodies recognised the same way; the
# kernel is inlined twice: lanes path and sequential fallback -- the three shortest loops with the right prefetch counts are taken)
ks = funcs[find('k_step_pitILi16ELi16ELi1E')[0]]
loops = []
for a, t in ks:
    m = re.search(r'BRA\s+(?:U?P\d,\s*)?(0x[0-9a-f]+)', t)
    if m and int(m.group(1), 16) < a:
        loops.append((int(m.group(1), 16), a))
b23 = sorted((l for l in loops if n_ldgsts(*l) == 23), key=lambda l: l[1] - l[0])
f14 = sorted((l for l in loops if n_ldgsts(*l) == 14), key=lambda l: l[1] - l[0])
if len(b23) >= 2 and f14:
    f = n = 0
    # shortest 23-field loop = plain in-chunk recursion, the longest = element pass (recursion + Gramian + closed-loop product)
    for lo, hi in (b23[0], b23[-1], f14[0]):
        a, b = flops(body(lo, hi)); f += a; n += b
    out['inst_step'] = {'flop_per_cell': f, 'instructions': n, 'note': 'k_step_pit<16,16>: element pass + in-chunk recursion + forward loop body per interval (chain steps not included)'}
json.dump(out, open(os.path.join(ROOT, 'profiles', 'fp64_ops.json'), 'w'), indent=1)
print(json.dumps(out, indent=1))
