import os, sys, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
from oracle import fdcm_oracle as orc
BIG = 0xFFFF
def fdiv(N, D): return N // D
class Stack:
    def __init__(s): s.e = []   # entries [key, v, bound]
    def take_over(s, v, key, Wm1):
        while s.e:
            tk, tv, ts = s.e[-1]
            N = key - tk; Dn = 2 * (v - tv)
            if N < ts * Dn: s.e.pop(); continue
            if N >= Wm1 * Dn: return Wm1 + 1
            return fdiv(N, Dn) + 1
        return 0
    def column(s, v, g, Wm1):
        key = g * g + v * v
        st = s.take_over(v, key, Wm1)
        if st <= Wm1: s.e.append([key, v, st])
    def column_rev(s, v, g, Wm1):
        key = g * g + v * v; end = Wm1
        while s.e:
            tk, tv, ts = s.e[-1]
            N = tk - key; Dn = 2 * (tv - v)
            if N >= ts * Dn: s.e.pop(); continue
            if N < 0: return
            end = fdiv(N, Dn); break
        s.e.append([key, v, end])
def join_right(st, right, Wm1):
    j = 0; rs = 0
    while j < len(right):
        key, v, end = right[j]; j += 1
        start = st.take_over(v, key, Wm1)
        if start <= end:
            st.e.append([key, v, start]); rs = end + 1; break
    return j, rs
def envelope4(g, x1, x2, x3):
    n = len(g); Wm1 = n - 1
    S = [Stack() for _ in range(4)]
    for v in range(0, x1):
        if g[v] != BIG: S[0].column(v, int(g[v]), Wm1)
    for v in range(x2 - 1, x1 - 1, -1):
        if g[v] != BIG: S[1].column_rev(v, int(g[v]), Wm1)
    for v in range(x2, x3):
        if g[v] != BIG: S[2].column(v, int(g[v]), Wm1)
    for v in range(n - 1, x3 - 1, -1):
        if g[v] != BIG: S[3].column_rev(v, int(g[v]), Wm1)
    r1 = S[1].e[::-1]; r3 = S[3].e[::-1]       # ascending v
    used, rs01 = join_right(S[0], r1, Wm1)
    start = rs01
    for (key, v, end) in r1[used:]:
        S[0].e.append([key, v, start]); start = end + 1
    used3, rs23 = join_right(S[2], r3, Wm1)
    L23 = list(S[2].e); R23 = r3[used3:]
    kl, kr = len(L23), len(R23)
    i = 0; found = False; start = 0
    while i < kl + kr:
        if i < kl:
            key, v, _ = L23[i]
            end = L23[i + 1][2] - 1 if i + 1 < kl else (rs23 - 1 if kr > 0 else Wm1)
        else:
            key, v, end = R23[i - kl]
        start = S[0].take_over(v, key, Wm1)
        if start <= end: found = True; break
        i += 1
    ent = [(k, v, s) for k, v, s in S[0].e]     # (key, v, start)
    if found:
        if i < kl:
            ent.append((L23[i][0], L23[i][1], start))
            ent += [(k, v, s) for k, v, s in L23[i + 1:]]
            s2 = rs23
            for (k, v, e) in R23:
                ent.append((k, v, s2)); s2 = e + 1
        else:
            s2 = start
            for (k, v, e) in R23[i - kl:]:
                ent.append((k, v, s2)); s2 = e + 1
    return ent
def fill(ent, n):
    out = np.zeros(n, np.float64)
    if not ent: return np.full(n, np.finfo(np.float32).max)
    base = []
    for k, (key, v, s) in enumerate(ent):
        f = key - v * v
        if s > v:
            j = k - 1
            while ent[j][2] > v: j -= 1
            f = base[j] + (v - ent[j][1]) ** 2
        base.append(f)
    k = 0
    for q in range(n):
        while k + 1 < len(ent) and ent[k + 1][2] <= q: k += 1
        out[q] = base[k] + (q - ent[k][1]) ** 2
    return out
rng = np.random.default_rng(0)
bad = 0
for trial in range(3000):
    n = int(rng.integers(1, 400))
    mode = trial % 6
    g = rng.integers(0, [3, 10, 50, 400, 2800, 40][mode], n)
    if trial % 3 == 0: g = np.where(rng.random(n) < 0.7, BIG, g)
    if trial % 7 == 0: g = np.where(np.arange(n) < n // 3, g, BIG)
    if trial % 11 == 0: g = np.where(np.arange(n) > 2 * n // 3, g, BIG)
    x2 = int(rng.integers(0, n + 1)); x1 = int(rng.integers(0, x2 + 1)); x3 = int(rng.integers(x2, n + 1))
    ent = envelope4(g, x1, x2, x3)
    got = fill(ent, n).astype(np.float32)
    fmax = np.finfo(np.float32).max
    f = np.where(g == BIG, fmax, g.astype(np.float64) ** 2).astype(np.float32)
    want = orc.dt_pass_l2_1d(f)
    if not np.array_equal(got, want):
        bad += 1
        if bad < 4: print("MISMATCH trial", trial, n, x1, x2, x3, np.flatnonzero(got != want)[:5])
print("bad", bad)
