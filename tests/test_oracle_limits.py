"""CPU: the C oracle (oracle/ascore_oracle.c) at the shapes tests/test_gpu_limits.py scores, against things that do
not share its code -- a real libstdc++ std::unordered_map for the tie order, a float64 / exact binomial tail for the
score table, closed-form fragment counts.  The oracle was only compared with the compiled reference on ordinary
shapes (tests/golden/oracle_vs_ref.json); these checks make it a trustworthy yardstick at the limits the library
promises (include/pyascore_b200.h)."""
import ctypes as C
import itertools
import math
import shutil
import subprocess
from decimal import Context, Decimal

import numpy as np
import pytest

import _limits
from oracle.cscorer import OraclePyAscore, lib

HASH_PROBE = r"""
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <unordered_map>
#include <vector>
// o: keys (int64, binary) on stdin -> the iteration order of an unordered_map<long, uint32_t> they were inserted into
// c N: the bucket counts a map passes through while N elements are inserted one by one (_Prime_rehash_policy)
int main(int argc, char** argv) {
    if (argv[1][0] == 'o') {
        long n;
        if (fread(&n, sizeof(n), 1, stdin) != 1) return 1;
        std::vector<long> keys(n);
        if (fread(keys.data(), sizeof(long), n, stdin) != (size_t)n) return 1;
        std::unordered_map<long, uint32_t> m;
        for (long i = 0; i < n; i++) m[keys[i]] = (uint32_t)i;
        for (auto& kv : m) fwrite(&kv.first, sizeof(long), 1, stdout);
        return 0;
    }
    const long N = atol(argv[2]);
    std::__detail::_Prime_rehash_policy pol;
    std::size_t n_bkt = 1;
    for (long e = 0; e < N; e++) {
        auto r = pol._M_need_rehash(n_bkt, (std::size_t)e, 1);
        if (r.first) { n_bkt = r.second; printf("%ld %zu\n", e, n_bkt); }
    }
    // the same on a real container, as far as memory allows
    std::unordered_map<long, uint32_t> m;
    std::size_t last = m.bucket_count();
    for (long e = 0; e < (N < 3000000 ? N : 3000000); e++) {
        m[e] = 0;
        if (m.bucket_count() != last) { last = m.bucket_count(); printf("real %ld %zu\n", e, last); }
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def hash_probe(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("hash_probe")
    src, exe = d / "probe.cpp", d / "probe"
    src.write_text(HASH_PROBE)
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-o", str(exe), str(src)])
    return str(exe)


def combination_keys(S, k, forward):
    """the oracle's insertion order (enumerate_keys): k-combinations of traversal positions in lexicographic order,
    site j of the peptide (N->C) at bit S-1-j"""
    keys = np.empty(math.comb(S, k), np.int64)
    for q, c in enumerate(itertools.combinations(range(S), k)):
        key = 0
        for t in c:
            site = t if forward else S - 1 - t
            key |= 1 << (S - 1 - site)
        keys[q] = key
    return keys


def oracle_hash_order(keys):
    L = lib("orc_")
    f = L._dll.orc_hash_order
    f.argtypes = [C.c_void_p, C.c_long, C.c_void_p]
    k = np.ascontiguousarray(keys.astype(np.uint64))
    order = np.zeros(k.size, np.int64)
    f(k.ctypes.data, k.size, order.ctypes.data)
    return keys[order]


@pytest.mark.parametrize("S,k", [(20, 1), (20, 3), (32, 1), (32, 2), (32, 3), (33, 1), (33, 2), (33, 3), (48, 1),
                                 (48, 2), (48, 3), (63, 1), (63, 2), (63, 3), (63, 4)])
def test_hash_order_matches_libstdcxx(hash_probe, S, k):
    """the oracle's model of the iteration order of unordered_map<long, ...> (which decides the order of tied
    isoforms) equals the real container for signatures of 33..63 bits, both enumeration directions, up to
    C(63, 4) = 595 665 keys"""
    for forward in ((True, False) if k < 4 else (True,)):
        keys = combination_keys(S, k, forward)
        inp = np.int64(keys.size).tobytes() + keys.tobytes()
        out = subprocess.run([hash_probe, "o"], input=inp, stdout=subprocess.PIPE, check=True).stdout
        real = np.frombuffer(out, np.int64)
        model = oracle_hash_order(keys)
        assert real.size == keys.size
        first = int(np.argmax(real != model)) if not np.array_equal(real, model) else -1
        assert first < 0, "S=%d k=%d forward=%s: order differs from position %d of %d" % (S, k, forward, first, keys.size)


def test_bucket_chain_covers_isoform_limit(hash_probe):
    """the bucket counts the oracle's model steps through (BKT_CHAIN) are those of libstdc++'s rehash policy for every
    element count up to the largest isoform count the library scores (PA_MAX_ISOFORMS = 2^26), and the real container
    agrees for the first three million insertions"""
    n_max = _limits.MAX_ISOFORMS + 1
    out = subprocess.run([hash_probe, "c", str(n_max)], stdout=subprocess.PIPE, check=True, text=True).stdout
    policy, real = [], []
    for line in out.splitlines():
        f = line.split()
        (real if f[0] == "real" else policy).append((int(f[-2]), int(f[-1])))
    chain = np.zeros(64, np.uint64)
    f = lib("orc_")._dll.orc_bkt_chain
    f.restype = C.c_long
    f.argtypes = [C.c_void_p, C.c_long]
    n = f(chain.ctypes.data, chain.size)
    chain = [int(x) for x in chain[:n]]
    # the model rehashes before inserting element e when e + 1 exceeds the current bucket count
    assert policy[0][0] == 0
    assert [b for _, b in policy] == chain[:len(policy)]
    assert [e for e, _ in policy[1:]] == chain[:len(policy) - 1]
    assert chain[len(policy) - 1] >= _limits.MAX_ISOFORMS          # the last step holds 2^26 elements
    assert real == policy[:len(real)] and len(real) >= 17


def _exact_tail_scores(n, p):
    """|-10 log10 P(X >= k)|, X ~ Binomial(n, p), k = 0..n, from the exact sum of the pmf in 50-digit decimal
    arithmetic (no underflow: the exponent range is unbounded for these sizes)"""
    ctx = Context(prec=50, Emin=-10 ** 9, Emax=10 ** 9)
    P = Decimal(p)
    Q = ctx.subtract(Decimal(1), P)
    term = ctx.power(P, n)
    acc = Decimal(0)
    out = np.zeros(n + 1)
    for j in range(n, 0, -1):
        acc = ctx.add(acc, term)
        out[j] = float(ctx.multiply(Decimal(-10), ctx.log10(acc)))
        term = ctx.divide(ctx.multiply(ctx.multiply(term, Decimal(j)), Q), ctx.multiply(Decimal(n - j + 1), P))
    return np.abs(out)


# |oracle - float64 reference| / max(reference, 1) measured on rows 1 .. 4095 (those sampled below), all ten depths:
# one float32 rounding (<= 8.3e-8) on short rows, then a drift that grows with n -- 2.7e-5 at mz_error 0.02
# (1.3e-8 x n at n = 2048), 0.0045 at 0.5 (1.09e-6 x n at n = 4094), 0.0135 at 1.5 (6.6e-6 x n at n = 2049).  It is
# the drift of the reference's float32 log-sum recursion, which the oracle restates on purpose.  The bound is
# TAIL_REL_ROUND + TAIL_REL_PER_TRIAL[mz_error] x n, with 1.5x headroom on each part; a wrong log-table index, an
# overflowing row offset or a recursion that runs off grows far past it.
TAIL_REL_ROUND = 1.2e-7
TAIL_REL_PER_TRIAL = {0.02: 2e-8, 0.5: 1.6e-6, 1.5: 1.0e-5}


@pytest.mark.parametrize("err", sorted(TAIL_REL_PER_TRIAL))
def test_score_table_against_binomial_tail(err):
    from scipy.stats import binom
    L = lib("orc_")._dll
    L.orc_new.restype = C.c_void_p
    L.orc_new.argtypes = [C.c_float, C.c_size_t, C.c_char_p, C.c_float, C.c_float, C.c_char_p]
    L.orc_depth_score.restype = C.c_float
    L.orc_depth_score.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t]
    L.orc_free.argtypes = [C.c_void_p]
    h = L.orc_new(100., 10, b"STY", 79.966331, err, b"by")
    rng = np.random.default_rng(int(err * 10))
    rows = [1, 2, 10, 100, 512, 1025, 2048, 2049, 4094, 4095] + rng.integers(101, 4095, 1).tolist()
    try:
        for n in rows:
            for d in range(10):
                # cpp/Ascore.cpp:23-36: p_d = 2 * err * d / 100 in the reference's float / double steps
                p = float(np.float32(float(np.float32(np.float32(2 * np.float32(err)) * np.float32(d + 1))) / 100.))
                got = np.array([L.orc_depth_score(h, d, k, n) for k in range(n + 1)], np.float64)
                ls = binom.logsf(np.arange(n + 1) - 1, n, p)
                ref = np.abs(-10. * ls / np.log(10.))
                under = ~np.isfinite(ls) | (ls < -700.)
                if under.any():
                    ex = _exact_tail_scores(n, p)
                    ref[under] = ex[under]
                    ok = ~under & (ref > 1e-3)
                    assert np.all(np.abs(ex[ok] - ref[ok]) <= 1e-9 * ref[ok])     # the two references agree
                rel = np.abs(got - ref) / np.maximum(ref, 1.)
                assert rel.max() <= TAIL_REL_ROUND + TAIL_REL_PER_TRIAL[err] * n, (n, d, int(np.argmax(rel)), rel.max())
    finally:
        L.orc_free(h)


def test_fragment_counts_closed_form():
    """total_fragments of every isoform the oracle scores at the limit shapes equals the closed form the library's
    fragment budget rests on: per ion type (L - 1) steps x charges x neutral-loss variants, one step with one variant
    fewer on a one-residue peptide"""
    groups = [f() for f in (_limits.length_group, lambda: _limits.length_group([("st", 97.9769)]), _limits.charge_group,
                            lambda: _limits.charge_group([("ST", 18.01528)]), _limits.frag_group, _limits.frag_group_nl,
                            _limits.dense_group)]
    for g in groups:
        sc = g.meta["scorer"]
        nl = {}
        for grp, m in g.meta["neutral_losses"]:
            for c in grp:
                nl[c] = m
        O = OraclePyAscore(**sc)
        for grp, m in g.meta["neutral_losses"]:
            O.add_neutral_loss(grp, m)
        for p, inf in zip(g.psms, g.info):
            O.score(p["mz"], p["inten"], p["peptide"], p["n_mod"], p["max_charge"])
            sig, cnt, scores, w, tot = O.pep_score_tables()
            pos = [i for i, c in enumerate(p["peptide"]) if c in sc["mod_group"]]
            for q in range(w.size):
                state = np.zeros(len(p["peptide"]), int)
                state[[pos[j] for j in range(len(pos)) if sig[q, j]]] = 1
                want = _limits.fragments_per_isoform(p["peptide"], state, sc["fragment_types"], p["max_charge"], nl)
                assert tot[q] == want, (g.name, p["peptide"], q, tot[q], want)
            if "n_frag" in inf:
                assert np.all(tot == inf["n_frag"]), (g.name, inf, tot)
            assert np.all(cnt[:, -1] <= tot)


def test_variant_matrix_covers_every_instantiation():
    """the scorer set-ups tests/test_gpu_limits.py::test_variant_matrix scores select every k_count_score<HAS_NL, PAIR,
    EGH> instantiation at least twice (computed from the settings), exactly 0.5 stays on the EGH = false side, and
    every pair of settings occurs"""
    seen = {}
    for f, e, nl in _limits.VARIANTS:
        v = _limits.k2_instantiation(f, e, nl)
        seen[v] = seen.get(v, 0) + 1
    assert len(seen) == 8 and min(seen.values()) >= 2, seen
    assert not _limits.k2_instantiation("by", 0.5, [])[2] and _limits.k2_instantiation("by", _limits.ERR_ABOVE_HALF, [])[2]
    sizes = [len(_limits.FTYPES), len(_limits.ERRS), len(_limits.NLS)]
    for a, b in ((0, 1), (0, 2), (1, 2)):
        pairs = {((f, e, len(nl))[a], (f, e, len(nl))[b]) for f, e, nl in _limits.VARIANTS}
        assert len(pairs) == sizes[a] * sizes[b]
