"""String restatements of the reference CPU assembler's link graph and get_contig, next to the oracle's
py_build / py_all_contigs -- test infrastructure only.  tests/test_cpu_unitig_wide.py pins both to the outputs of
the unmodified reference (tests/golden/*.json: `links`, `get_contig`)."""
from oracle import _fw, _walk_forward, twin


def py_get_contig(d, km):
    """referenceAssembler.py:47-56: (string, list of k-mers) of the unitig through km, on the oracle's walk."""
    c_fw = _walk_forward(d, km)
    c_bw = _walk_forward(d, twin(km))
    if km in _fw(c_fw[-1]):
        c = c_fw
    else:
        c = [twin(x) for x in c_bw[-1:0:-1]] + c_fw
    return c[0] + "".join(x[-1] for x in c[1:]), c


def py_link_graph(contigs, k):
    """The link graph G of referenceAssembler.py:90-111 for a contig list, in the shape
    {i: ([(j, '+' | '-'), ...] after the last k-mer, [...] after twin(first k-mer))}.  A later contig
    overwrites an earlier one in heads / tails."""
    G, heads, tails = {}, {}, {}
    for i, x in enumerate(contigs):
        G[i] = ([], [])
        heads[x[:k]] = (i, "+")
        tails[twin(x[-k:])] = (i, "-")
    for i in G:
        x = contigs[i]
        for side, km in ((0, x[-k:]), (1, twin(x[:k]))):
            for y in _fw(km):
                if y in heads:
                    G[i][side].append(heads[y])
                if y in tails:
                    G[i][side].append(tails[y])
    return G
