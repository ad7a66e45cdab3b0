#!/bin/bash
# multi-GPU partition driver == single-GPU assembly (run under: gpurun --gpus 2 -- bash scripts/check_assembler.sh 2)
set -e
N=${1:-2}
cd "$(dirname "$0")/.."
python - <<'PY'
import sys
sys.path.insert(0, '.')
import oracle
G, L, cov = 300000, 100, 25
n = G * cov // L
r = oracle.synth_reads(G, L, err_ppm=3000, first=0, count=n)
with open('/tmp/reads.fq', 'wb') as f:
    for i in range(n):
        s = bytes(r[i * L:(i + 1) * L])
        f.write(b'@r%d\n%s\n+\n%s\n' % (i, s, b'I' * L))
PY
python pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/one.fa -k 31
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29531 \
    pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/multi.fa -k 31
python - <<'PY'
def canon(path):
    comp = str.maketrans('ACGT', 'TGCA')
    out = []
    for line in open(path):
        if line[0] != '>':
            c = line.strip()
            out.append(min(c, c.translate(comp)[::-1]))
    return sorted(out)
a, b = canon('/tmp/one.fa'), canon('/tmp/multi.fa')
print('single-GPU contigs', len(a), 'multi-GPU contigs', len(b), 'equal sets:', a == b)
assert a == b and len(a) > 0
print('gfa links:', sum(1 for l in open('/tmp/multi.fa.gfa') if l[0] == 'L'), 'vs', sum(1 for l in open('/tmp/one.fa.gfa') if l[0] == 'L'))
PY
# --clean: the contig set of one assembly across GPUs (clean-up on the joined table) equals the single-GPU one
python pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/one_c.fa -k 31 --clean
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 \
    pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/multi_c.fa -k 31 --clean
python - <<'PY'
def canon(path):
    comp = str.maketrans('ACGT', 'TGCA')
    return sorted(min(c, c.translate(comp)[::-1]) for c in (l.strip() for l in open(path)) if c and c[0] != '>')
a, b = canon('/tmp/one_c.fa'), canon('/tmp/multi_c.fa')
print('--clean: single-GPU contigs', len(a), 'multi-GPU contigs', len(b), 'equal sets:', a == b)
assert a == b and len(a) > 0
PY
# Euler mode: identical contig LIST (canonical ids make the tour deterministic)
python pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/one_e.fa -k 32 --mode euler
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29532 \
    pycuda-euler_b200/assembler.py -i /tmp/reads.fq -o /tmp/multi_e.fa -k 32 --mode euler
cmp /tmp/one_e.fa /tmp/multi_e.fa && echo "euler mode: identical output ($(grep -c '>' /tmp/one_e.fa) contigs)"
