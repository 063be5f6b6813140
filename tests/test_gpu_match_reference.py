"""M1 SMNN matching (csrc/match_tc.cu, csrc/match.cu) against a float64 reference, on both distance kernels.

The GPU decides on fp32 distances, so near-ties can legitimately go either way.  Instead of a tolerance on the output, the
tests bound the kernel's error E on every squared distance, |d_gpu^2 - d64^2| <= E * (|a|^2 + |b|^2), and classify each
row from float64 distances with interval reasoning:

* certainly matched: the nearest neighbour holds in both directions and both ratio tests hold for every distance within
  +-E (plus one rounding of the fp32 ratio);
* certainly unmatched: no pair of the row can be output for any such distances;
* undetermined: everything else.

The GPU output must contain every certainly-matched pair and only pairs that are possible.  To keep that sensitive, the
near-tie set has to leave at least 80 % of its rows determined.  Decisions that do not depend on rounding (tie rule,
threshold comparison, direction symmetry) are checked bit for bit against oracle.thirdparty.match_smnn on the GPU's own
distance matrix.  The distance kernel is switched with balf_debug_set(3, impl): 0 = 3xTF32 tensor cores, 1 = fp32 FFMA.
"""
import math

import numpy as np
import pytest
import torch

from oracle import thirdparty

gpu = pytest.mark.gpu

PATHS = {"tc": 0, "ffma": 1}
# E: bound on |d_gpu^2 - d64^2| / (|a|^2 + |b|^2), about 2x the maximum measured over this file's inputs on an NVIDIA
# B200 (1000 W power limit): 3xTF32 tensor cores 1.95e-6, fp32 FFMA 6.4e-7.  The tensor-core path is the less accurate
# one: its fp32 accumulation truncates.
E_BOUND = {"tc": 4e-6, "ffma": 1.5e-6}
RATIO_SLACK = 2.0 ** -22                  # the fp32 division v0 / v1 rounds once (2^-24); a 4x margin
TH_BELOW_1 = float(np.nextafter(np.float32(1.0), np.float32(0.0)))
GRID = 2.0 ** -20                         # near-tie coordinates are multiples of GRID: exact in fp32, exact d^2 in float64
DECADES = list(range(-8, -3))             # margin decades 1e-8 .. 1e-3 of the near-tie rows


def dev():
    return torch.device("cuda:0")


def capi():
    import balf_b200._capi as c
    return c


def run(path, d1, d2, th, want_dm=True):
    """balf_match_smnn on the chosen distance kernel -> (dist [M] fp32, ids [M,2] int64, dm or None), on the host."""
    c = capi()
    c.debug_set(3, PATHS[path])
    try:
        out = c.match_smnn(torch.as_tensor(d1).to(dev()), torch.as_tensor(d2).to(dev()), th, want_dm=want_dm)
    finally:
        c.debug_set(3, 0)
    dist, ids = out[0].cpu().numpy()[:, 0], out[1].cpu().numpy()
    return dist, ids, (out[2] if want_dm else None)


# ------------------------------------------------------------------------------------------ inputs
def correlated(n1, n2, seed, noise=0.15):
    """unit rows; about half of d2 are noisy copies of d1 rows, so that mutual matches exist"""
    g = torch.Generator().manual_seed(seed)
    d1 = torch.randn(n1, 128, generator=g, dtype=torch.float64)
    d2 = torch.randn(n2, 128, generator=g, dtype=torch.float64)
    m = min(n1, n2) // 2
    d2[:m] = d1[torch.randperm(n1, generator=g)[:m]] + noise * torch.randn(m, 128, generator=g, dtype=torch.float64) / 8
    d2 = d2[torch.randperm(n2, generator=g)]
    return ((d1 / d1.norm(dim=1, keepdim=True)).float().numpy(), (d2 / d2.norm(dim=1, keepdim=True)).float().numpy())


def _mirror_triple(rng, center, m_target=None, ratio=None, d0_range=(0.1, 0.4)):
    """integer (grid) rows (partner, rival) around `center`: the rival mirrors the partner through the centre, which ties
    the two distances exactly, then one coordinate moves the rival away by a chosen margin (in GRID^2 units):
    margin = 2 k delta + k^2.  With `ratio` the margin makes d(partner) / d(rival) = ratio instead."""
    d0 = rng.uniform(*d0_range)
    partner = center + np.rint(rng.standard_normal(128) * math.sqrt(d0 / 128) / GRID).astype(np.int64)
    c = int(rng.integers(128))
    approx = m_target / GRID ** 2 if ratio is None else d0 * (1 / ratio ** 2 - 1) / GRID ** 2
    delta = max(1, int(round(math.sqrt(approx / 3))))
    partner[c] = center[c] + delta
    if ratio is not None:
        d0_exact = int(((partner - center) ** 2).sum())
        m_units = d0_exact * (1 / ratio ** 2 - 1)
    else:
        m_units = m_target / GRID ** 2
    k = max(1, int(math.ceil(-delta + math.sqrt(delta * delta + m_units))))     # margin >= the target
    rival = 2 * center - partner
    rival[c] -= k
    return partner, rival


def near_tie_set(seed=7, n_tie=512, n_ratio=1024, n_plain=4096, th=0.99):
    """Queries d1 and keys d2 (fp32, near unit norm) with near-ties on both sides:
    - n_tie queries whose nearest key has a rival key at a squared-distance margin log-uniform in 1e-8 .. 1e-3;
    - n_tie keys whose nearest query has a rival query at such a margin;
    - n_ratio queries whose float64 ratio d(nearest) / d(second) lies within +-1e-4 of th (at least 10^-5.5 away, and
      with a far nearest neighbour, so that most of them stay determined under the tensor-core bound);
    - n_plain query / key pairs without a rival.
    Every coordinate is a multiple of 2^-20, so the fp32 rows hold the intended margins exactly.  Returns (d1, d2, meta)
    with the intended (query or key index, margin or ratio) of every constructed row."""
    rng = np.random.default_rng(seed)

    def unit():
        v = rng.standard_normal(128)
        return np.rint(v / np.linalg.norm(v) / GRID).astype(np.int64)

    Q, K, q_ties, k_ties, q_ratio = [], [], [], [], []
    for _ in range(n_tie):                                    # query with two keys
        m = 10.0 ** rng.uniform(-8, -3)
        c = unit()
        a, b = _mirror_triple(rng, c, m_target=m)
        q_ties.append((len(Q), len(K), len(K) + 1))
        Q.append(c); K += [a, b]
    for _ in range(n_tie):                                    # key with two queries
        m = 10.0 ** rng.uniform(-8, -3)
        c = unit()
        a, b = _mirror_triple(rng, c, m_target=m)
        k_ties.append((len(K), len(Q), len(Q) + 1))
        K.append(c); Q += [a, b]
    for _ in range(n_ratio):
        r = th + rng.choice([-1.0, 1.0]) * 10.0 ** rng.uniform(-5.5, -4)
        c = unit()
        a, b = _mirror_triple(rng, c, ratio=r, d0_range=(0.6, 0.9))
        q_ratio.append((len(Q), len(K), len(K) + 1))
        Q.append(c); K += [a, b]
    for _ in range(n_plain):
        c = unit()
        d0 = rng.uniform(0.1, 0.4)
        Q.append(c); K.append(c + np.rint(rng.standard_normal(128) * math.sqrt(d0 / 128) / GRID).astype(np.int64))
    pq, pk = rng.permutation(len(Q)), rng.permutation(len(K))    # spread the groups over tiles, CTAs and key splits
    iq, ik = np.argsort(pq), np.argsort(pk)                      # original index -> new index
    d1 = (np.array(Q, dtype=np.float64)[pq] * GRID).astype(np.float32)
    d2 = (np.array(K, dtype=np.float64)[pk] * GRID).astype(np.float32)
    meta = {"q_ties": np.array([(iq[a], ik[b], ik[c]) for a, b, c in q_ties]),
            "k_ties": np.array([(ik[a], iq[b], iq[c]) for a, b, c in k_ties]),
            "q_ratio": np.array([(iq[a], ik[b], ik[c]) for a, b, c in q_ratio]), "th": th}
    return d1, d2, meta


def scaled_norms(d1, d2, seed):
    """rows scaled to norms log-uniform in [0.1, 10]; partners keep their partner's scale to within a few percent"""
    rng = np.random.default_rng(seed)
    s1 = 10.0 ** rng.uniform(-1, 1, len(d1))
    nn = np.argmax(d2.astype(np.float64) @ d1.astype(np.float64).T, axis=1)      # best-aligned query of every key
    s2 = np.clip(s1[nn] * np.exp(0.03 * rng.standard_normal(len(d2))), 0.1, 10)
    free = rng.random(len(d2)) < 0.25                                            # some keys get a scale of their own
    s2[free] = 10.0 ** rng.uniform(-1, 1, int(free.sum()))
    return (d1 * s1[:, None]).astype(np.float32), (d2 * s2[:, None]).astype(np.float32)


# ------------------------------------------------------------------------------------------ float64 reference
def sqdist64(a, b):
    """float64 squared distances |a|^2 + |b|^2 - 2 a.b of fp32 rows (NumPy)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return (a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * (a @ b.T)


def _row_stats(d2, s, E):
    """per row: the two smallest squared distances with indices, and the two smallest of their lower / upper bounds"""
    dv, di = torch.topk(d2, 2, dim=1, largest=False)
    lv, li = torch.topk(d2 - E * s, 2, dim=1, largest=False)
    uv, _ = torch.topk(d2 + E * s, 2, dim=1, largest=False)
    return [dv, di, lv, li, uv]


def _merge_cols(run_, new, offset):
    """merge the column statistics of a row chunk (indices relative to it) into the running ones"""
    new = list(new)
    new[1] = new[1] + offset
    new[3] = new[3] + offset
    if run_ is None:
        return new
    out = []
    for (v, i), (nv, ni) in (((run_[0], run_[1]), (new[0], new[1])), ((run_[2], run_[3]), (new[2], new[3]))):
        cv, ci = torch.cat([v, nv], 1), torch.cat([i, ni], 1)
        o = torch.argsort(cv, dim=1, stable=True)[:, :2]
        out += [cv.gather(1, o), ci.gather(1, o)]
    uv = torch.sort(torch.cat([run_[4], new[4]], 1), dim=1).values[:, :2]
    return out + [uv]


class Reference:
    """float64 row and column summaries of the squared-distance matrix of d1 x d2 and the certainty classification for a
    kernel error bound E.  Rows are processed in chunks, on `device`, with running column top-2s."""

    def __init__(self, d1, d2, E, device="cpu", chunk=4096):
        a = torch.as_tensor(d1).to(device).double()
        b = torch.as_tensor(d2).to(device).double()
        self.a, self.b, self.E = a, b, E
        self.na, self.nb = (a * a).sum(1), (b * b).sum(1)
        rows, cols = [], None
        for r0 in range(0, len(a), chunk):
            ac = a[r0:r0 + chunk]
            d2m = self.na[r0:r0 + chunk, None] + self.nb[None, :] - 2.0 * (ac @ b.T)
            s = self.na[r0:r0 + chunk, None] + self.nb[None, :]
            rows.append(_row_stats(d2m, s, E))
            cols = _merge_cols(cols, _row_stats(d2m.T, s.T, E), r0)
            del d2m, s
        self.rows = [torch.cat([r[k] for r in rows]) for k in range(5)]
        self.cols = cols

    def pair_d2(self, i, j):
        i, j = torch.as_tensor(i, device=self.a.device), torch.as_tensor(j, device=self.a.device)
        return self.na[i] + self.nb[j] - 2.0 * (self.a[i] * self.b[j]).sum(1)

    def _side(self, stats, n_self, n_other, th):
        dv, di, lv, li, uv = stats
        nn = di[:, 0]
        s_nn = n_self + n_other[nn]
        lo_other = torch.where(li[:, 0] != nn, lv[:, 0], lv[:, 1])          # smallest lower bound of any other candidate
        cert = dv[:, 0] + self.E * s_nn < lo_other
        lo0, lo1 = lv[:, 0].clamp(min=0), lv[:, 1].clamp(min=0)
        r_lo = torch.where(uv[:, 1] > 0, torch.sqrt(lo0 / uv[:, 1].clamp(min=1e-300)), torch.zeros_like(lo0)) * (1 - RATIO_SLACK)
        r_hi = torch.where(lo1 > 0, torch.sqrt(uv[:, 0] / lo1.clamp(min=1e-300)) * (1 + RATIO_SLACK),
                           torch.full_like(lo0, math.inf))
        r_hi = torch.where(lo1 > 0, r_hi.clamp(max=1.0), r_hi)             # v0 <= v1 and v1 > 0: the fp32 ratio is <= 1
        return {"nn": nn, "cert": cert, "minup": uv[:, 0], "r_lo": r_lo, "r_hi": r_hi, "lo_nn": dv[:, 0] - self.E * s_nn,
                "margin": dv[:, 1] - dv[:, 0]}

    def classify(self, th):
        """-> (row side, column side, certainly matched pairs [P,2] int64 numpy); each side also carries `determined`"""
        R, C = self._side(self.rows, self.na, self.nb, th), self._side(self.cols, self.nb, self.na, th)
        for X, Y in ((R, C), (C, R)):
            other = X["nn"]
            X["pass"] = (X["r_hi"] <= th) & (Y["r_hi"][other] <= th)
            X["impossible"] = (X["lo_nn"] > Y["minup"][other]) | (X["r_lo"] > th) | (Y["r_lo"][other] > th)
        ar = torch.arange(len(R["nn"]), device=self.a.device)
        matched = R["cert"] & C["cert"][R["nn"]] & (C["nn"][R["nn"]] == ar) & R["pass"]
        C["matched"] = torch.zeros_like(C["cert"])
        C["matched"][R["nn"][matched]] = True
        R["matched"] = matched
        for X in (R, C):
            X["determined"] = (X["cert"] & (X["matched"] | X["impossible"])) | (X["r_lo"] > th)
        pairs = torch.stack([ar[matched], R["nn"][matched]], 1)
        return R, C, pairs.cpu().numpy()

    def check(self, ids, dist, th):
        """the GPU output (ids [M,2], dist [M]) against the certainty rule; returns the classification"""
        R, C, pairs = self.classify(th)
        ids = np.asarray(ids).reshape(-1, 2)
        assert np.all(np.diff(ids[:, 0]) > 0), "ids must be strictly ascending in the first index"
        got = set(map(tuple, ids.tolist()))
        missing = [p for p in map(tuple, pairs.tolist()) if p not in got]
        assert not missing, "%d certainly-matched pairs missing, e.g. %s" % (len(missing), missing[:5])
        if len(ids):
            i = torch.as_tensor(ids[:, 0], device=self.a.device)
            j = torch.as_tensor(ids[:, 1], device=self.a.device)
            lo = self.pair_d2(i, j) - self.E * (self.na[i] + self.nb[j])
            ok = (lo <= R["minup"][i]) & (lo <= C["minup"][j]) & (R["r_lo"][i] <= th) & (C["r_lo"][j] <= th)
            bad = (~ok).nonzero().flatten().cpu().numpy()
            assert len(bad) == 0, "%d impossible pairs in the output, e.g. %s" % (len(bad), ids[bad[:5]].tolist())
            lo_d = torch.maximum(R["r_lo"][i], C["r_lo"][j]).cpu().numpy()
            hi_d = torch.maximum(R["r_hi"][i], C["r_hi"][j]).cpu().numpy()
            d = np.asarray(dist, np.float64)
            assert np.all((d >= lo_d) & (d <= hi_d)), "dist outside the float64 ratio bounds at rows %s" % \
                ids[~((d >= lo_d) & (d <= hi_d)), 0][:5]
        return R, C, pairs


def max_rel_err(dm, d1, d2):
    """max over the matrix of |dm^2 - d64^2| / (|a|^2 + |b|^2), computed in row chunks on dm's device"""
    a = torch.as_tensor(np.asarray(d1), device=dm.device).double()
    b = torch.as_tensor(np.asarray(d2), device=dm.device).double()
    na, nb = (a * a).sum(1), (b * b).sum(1)
    worst = 0.0
    for r0 in range(0, len(a), 4096):
        ref = na[r0:r0 + 4096, None] + nb[None] - 2.0 * (a[r0:r0 + 4096] @ b.T)
        err = (dm[r0:r0 + 4096].double() ** 2 - ref).abs() / (na[r0:r0 + 4096, None] + nb[None])
        worst = max(worst, float(err.max()))
    return worst


def oracle_bits(dist, ids, d1, d2, th, dm):
    """ids and dists bit-identical to thirdparty.match_smnn on the GPU's distance matrix"""
    want_dist, want_ids = thirdparty.match_smnn(torch.as_tensor(d1), torch.as_tensor(d2), th, dm=dm.cpu())
    np.testing.assert_array_equal(ids, want_ids.numpy().reshape(-1, 2))
    np.testing.assert_array_equal(dist.view(np.uint32), want_dist.numpy().reshape(-1).astype(np.float32).view(np.uint32))


def sensitivity(R, C):
    """fraction of determined rows (both sides) and determined rows per margin decade"""
    det = torch.cat([R["determined"], C["determined"]]).cpu().numpy()
    margin = torch.cat([R["margin"], C["margin"]]).cpu().numpy()
    per = {}
    for e in DECADES:
        sel = (margin >= 10.0 ** e) & (margin < 10.0 ** (e + 1))
        per[e] = (int(det[sel].sum()), int(sel.sum()))
    return float(det.mean()), per


# ------------------------------------------------------------------------------------------ CPU: generator and reference
def test_near_tie_generator_margins():
    d1, d2, meta = near_tie_set()
    assert d1.dtype == d2.dtype == np.float32
    D = sqdist64(d1, d2)
    for key, DD in (("q_ties", D), ("k_ties", D.T)):
        t = meta[key]
        row = DD[t[:, 0]]
        srt = np.sort(row, 1)
        margin = row[np.arange(len(t)), t[:, 2]] - row[np.arange(len(t)), t[:, 1]]
        assert np.all(row.argmin(1) == t[:, 1])                                 # the partner is the nearest
        assert np.array_equal(srt[:, 1], row[np.arange(len(t)), t[:, 2]])       # the rival is the second
        assert np.all(srt[:, 2] - srt[:, 1] > 0.1)                              # everything else is far
        dec = np.floor(np.log10(margin))
        assert margin.min() >= 1e-8 * 0.9 and margin.max() < 1.1e-3
        for e in DECADES:                                                      # log-uniform: every decade populated
            assert (dec == e).sum() >= 0.12 * len(t), (key, e, (dec == e).sum())
        # the margin is exact: integer grid arithmetic agrees with float64 on the fp32 rows
        g = np.rint(np.asarray(d1 if key == "q_ties" else d2, np.float64)[t[:5, 0]] / GRID).astype(np.int64)
        o = np.rint(np.asarray(d2 if key == "q_ties" else d1, np.float64) / GRID).astype(np.int64)
        for r in range(5):
            mi = ((g[r] - o[t[r, 2]]) ** 2).sum() - ((g[r] - o[t[r, 1]]) ** 2).sum()
            assert mi * GRID ** 2 == margin[r]
    t = meta["q_ratio"]
    row = D[t[:, 0]]
    ratio = np.sqrt(row[np.arange(len(t)), t[:, 1]] / row[np.arange(len(t)), t[:, 2]])
    assert np.all(row.argmin(1) == t[:, 1])
    off = ratio - meta["th"]
    assert np.abs(off).max() <= 1e-4 and (off < 0).sum() > 0.4 * len(t) and (off > 0).sum() > 0.4 * len(t)
    assert np.abs(off).min() >= 10 ** -5.5 * 0.9 and (np.abs(off) < 1e-5).sum() > 0.1 * len(t)
    srt = np.sort(row, 1)
    assert np.array_equal(srt[:, 1], row[np.arange(len(t)), t[:, 2]]) and np.all(srt[:, 2] - srt[:, 1] > 0.1)


def test_reference_chunks_agree_with_numpy():
    d1, d2 = correlated(300, 257, 11)
    whole, chunked = Reference(d1, d2, 1e-6), Reference(d1, d2, 1e-6, chunk=37)
    for x, y in zip(whole.rows + whole.cols, chunked.rows + chunked.cols):
        if x.is_floating_point():
            torch.testing.assert_close(x, y, rtol=0, atol=1e-12)
        else:
            assert torch.equal(x, y)
    D = sqdist64(d1, d2)
    np.testing.assert_allclose(np.sort(D, 1)[:, :2], whole.rows[0].numpy(), rtol=0, atol=1e-12)
    np.testing.assert_allclose(np.sort(D, 0)[:2].T, whole.cols[0].numpy(), rtol=0, atol=1e-12)
    assert np.array_equal(D.argmin(1), whole.rows[1][:, 0].numpy())
    assert np.array_equal(D.argmin(0), whole.cols[1][:, 0].numpy())


def _emulated(d1, d2, th, noise, seed):
    """a stand-in GPU: match_smnn on float64 distances moved by up to `noise` * (|a|^2 + |b|^2), rounded to fp32"""
    D = sqdist64(d1, d2)
    s = (np.asarray(d1, np.float64) ** 2).sum(1)[:, None] + (np.asarray(d2, np.float64) ** 2).sum(1)[None]
    D = D + noise * s * np.random.default_rng(seed).uniform(-1, 1, D.shape)
    dm = torch.from_numpy(np.sqrt(np.maximum(D, 0)).astype(np.float32))
    dist, ids = thirdparty.match_smnn(torch.from_numpy(d1), torch.from_numpy(d2), th, dm=dm)
    return dist.numpy()[:, 0], ids.numpy()


@pytest.mark.parametrize("th", [1.0, 0.99])
def test_certainty_rule_accepts_bounded_errors_and_rejects_wrong_decisions(th):
    d1, d2, _ = near_tie_set(n_tie=128, n_ratio=128, n_plain=512)
    E = 5e-7
    ref = Reference(d1, d2, E)
    for seed in range(3):                                    # any output within the error bound passes
        dist, ids = _emulated(d1, d2, th, E / 2, seed)
        ref.check(ids, dist, th)
    dist, ids = _emulated(d1, d2, th, 0.0, 0)
    R, C, pairs = ref.classify(th)
    assert len(pairs) > 100
    keep = np.ones(len(ids), bool)
    keep[np.flatnonzero((ids[:, None] == pairs[None]).all(2).any(1))[0]] = False
    with pytest.raises(AssertionError, match="certainly-matched"):     # a dropped pair is caught
        ref.check(ids[keep], dist[keep], th)
    i = int(np.setdiff1d(np.arange(len(d1)), ids[:, 0])[0])         # an unmatched row paired with its farthest key
    at = int(np.searchsorted(ids[:, 0], i))
    bad_ids = np.insert(ids, at, [i, int(sqdist64(d1[i:i + 1], d2).argmax())], axis=0)
    with pytest.raises(AssertionError, match="impossible"):
        ref.check(bad_ids, np.insert(dist, at, 0.5), th)
    with pytest.raises(AssertionError, match="dist outside"):
        ref.check(ids, dist * (1 + 1e-3), th)
    dist, ids = _emulated(d1, d2, th, 1e-4, 0)                       # single-pass TF32-sized errors do not pass
    with pytest.raises(AssertionError):
        ref.check(ids, dist, th)


def test_wrappers_reject_cpu_tensors_without_a_device():
    c = capi()
    with pytest.raises(RuntimeError, match="CUDA"):
        c.match_smnn(torch.zeros(4, 128), torch.zeros(4, 128))
    with pytest.raises(RuntimeError, match="CUDA"):
        c.hardnet_forward(torch.zeros(2, 1, 32, 32), torch.zeros(1))
    with pytest.raises(RuntimeError, match="CUDA"):
        c.extract_patches_batch(torch.zeros(1, 40, 40, dtype=torch.uint8), torch.zeros(1, 3, 2), None, 60.0)


# ------------------------------------------------------------------------------------------ GPU: accuracy and certainty
@pytest.fixture(scope="module")
def tie_set():
    return near_tie_set()


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_distance_error_bound(path, tie_set):
    """|d_gpu^2 - d64^2| <= E (|a|^2 + |b|^2) on the near-tie set, on random unit rows and on non-unit rows"""
    d1, d2, _ = tie_set
    cases = [(d1, d2), correlated(2049, 1500, 3), scaled_norms(*correlated(1500, 2049, 4), 5)]
    worst = []
    for a, b in cases:
        _, _, dm = run(path, a, b, 0.99)
        worst.append(max_rel_err(dm, a, b))
    print("max |d^2 - d64^2| / (|a|^2 + |b|^2) on the %s path: %s" % (path, ["%.3g" % w for w in worst]))
    assert max(worst) <= E_BOUND[path], worst


@gpu
@pytest.mark.parametrize("th", [1.0, 0.99])
@pytest.mark.parametrize("path", list(PATHS))
def test_certainty_on_near_ties(path, th, tie_set):
    d1, d2, meta = tie_set
    dist, ids, dm = run(path, d1, d2, th)
    ref = Reference(d1, d2, E_BOUND[path], device=dev())
    R, C, pairs = ref.check(ids, dist, th)
    frac, per = sensitivity(R, C)
    print("%s th=%g: %.3f of rows determined; per margin decade (determined, rows): %s" % (path, th, frac, per))
    assert frac >= 0.8, frac
    if th == 1.0:
        s_max = float(torch.cat([ref.na, ref.nb]).max()) * 2
        for e, (n_det, _) in per.items():
            if 10.0 ** e > 2 * E_BOUND[path] * s_max:
                assert n_det >= 100, (e, per)
    else:                                                    # the rows whose float64 ratio is within 1e-4 of th
        q = torch.as_tensor(meta["q_ratio"][:, 0], device=dev())
        kept = int((R["determined"][q] & (R["r_hi"][q] <= th)).sum())
        dropped = int((R["determined"][q] & (R["r_lo"][q] > th)).sum())
        print("ratio rows within 1e-4 of th: %d certainly kept, %d certainly dropped of %d" % (kept, dropped, len(q)))
        assert kept >= 100 and dropped >= 100, (kept, dropped)


@gpu
@pytest.mark.parametrize("th", [1.0, 0.99])
@pytest.mark.parametrize("path", list(PATHS))
def test_directions_bit_identical(path, th, tie_set):
    """With th = 1 every row passes the ratio test, so each near-tie decision reaches the output: ids and dists equal the
    oracle's on the GPU's own (direction 1) distance matrix.  A distance that differed between the two directions by one
    ulp would change a mutual decision or a ratio in the dist column."""
    d1, d2, _ = tie_set
    dist, ids, dm = run(path, d1, d2, th)
    oracle_bits(dist, ids, d1, d2, th, dm)


@gpu
def test_paths_agree_on_determined_rows(tie_set):
    d1, d2, _ = tie_set
    for th in (1.0, 0.99):
        E = max(E_BOUND.values())
        R, C, _ = Reference(d1, d2, E, device=dev()).classify(th)
        out = {}
        for p in PATHS:
            _, ids, _ = run(p, d1, d2, th, want_dm=False)
            j = np.full(len(d1), -1)
            j[ids[:, 0]] = ids[:, 1]
            out[p] = j
        det = R["determined"].cpu().numpy()
        assert det.mean() >= 0.8
        np.testing.assert_array_equal(out["tc"][det], out["ffma"][det])


# ------------------------------------------------------------------------------------------ GPU: exact ties and thresholds
TIE_OFFSETS = (0, 1, 4, 64, 300, 1900)     # one FFMA thread, two FFMA slices, two 64-key tiles, TC key splits 0, 1 and 6


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_exact_ties_across_tiles_splits_and_slices(path):
    n, j0 = 2049, 40
    d1, d2 = correlated(n, n, 21, noise=0.5)
    rng = np.random.default_rng(22)
    tq, tk = 7, 11                                           # the query that sees tied keys, the key that sees tied queries
    rows_k = [j0 + o for o in TIE_OFFSETS]
    rows_q = [j0 + o for o in TIE_OFFSETS]
    v = d1[tq] + 0.05 * rng.standard_normal(128).astype(np.float32) / np.float32(8)
    d2[rows_k] = v / np.linalg.norm(v)
    w = d2[tk] + 0.05 * rng.standard_normal(128).astype(np.float32) / np.float32(8)
    d1[rows_q] = w / np.linalg.norm(w)
    D = sqdist64(d1, d2)
    assert set(np.flatnonzero(D[tq] == D[tq].min())) == set(rows_k)
    assert set(np.flatnonzero(D[:, tk] == D[:, tk].min())) == set(rows_q)
    for th in (1.0, TH_BELOW_1):
        dist, ids, dm = run(path, d1, d2, th)
        dm = dm.cpu().numpy()
        # a distance depends on the rows' contents, not on their positions (include/balf_b200.h: "Exactly equal distances
        # resolve to the lower index" needs exactly equal distances first)
        for r in rows_k[1:]:
            assert np.array_equal(dm[:, r].view(np.uint32), dm[:, rows_k[0]].view(np.uint32)), r
        for r in rows_q[1:]:
            assert np.array_equal(dm[r].view(np.uint32), dm[rows_q[0]].view(np.uint32)), r
        got = dict(map(tuple, ids.tolist()))
        if th == 1.0:                                        # ratio exactly 1 passes; the lowest index wins
            assert got.get(tq) == rows_k[0]
            assert got.get(rows_q[0]) == tk
            for r in rows_q[1:]:
                assert r not in got
            assert list(got.values()).count(rows_k[0]) == 1 and not set(rows_k[1:]) & set(got.values())
            assert dist[list(got).index(tq)] == 1.0 and dist[list(got).index(rows_q[0])] == 1.0
        else:                                                # ... and fails any th < 1
            assert tq not in got and not set(rows_q) & set(got)
            assert not set(rows_k) & set(got.values()) and tk not in got.values()
        oracle_bits(dist, ids, d1, d2, th, torch.from_numpy(dm))


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_threshold_boundary(path):
    d1, d2 = correlated(1000, 1200, 31, noise=0.5)
    dist, ids, dm = run(path, d1, d2, 1.0)
    assert len(ids) > 100
    oracle_bits(dist, ids, d1, d2, 1.0, dm)
    for k in (len(ids) // 3, len(ids) - 1):
        r = np.float32(dist[k])                                  # an exact fp32 ratio v0 / v1 of the GPU's distances
        assert 0 < r < 1
        for th, kept in ((float(r), True), (float(np.nextafter(r, np.float32(0))), False)):
            dd, ii, _ = run(path, d1, d2, th, want_dm=False)
            assert (tuple(ids[k]) in set(map(tuple, ii.tolist()))) == kept, (th, ids[k])
            oracle_bits(dd, ii, d1, d2, th, dm)
    dd, ii, _ = run(path, d1, d2, 1.5, want_dm=False)
    oracle_bits(dd, ii, d1, d2, 1.5, dm)
    np.testing.assert_array_equal(ii, ids)                      # above 1 the ratio test keeps everything th = 1 keeps


# ------------------------------------------------------------------------------------------ GPU: shapes
SIZES = (2, 3, 63, 64, 65, 127, 128, 129, 255, 256, 257, 2049)


def check_shape(path, n1, n2, seed, th=0.99):
    d1, d2 = correlated(n1, n2, seed)
    dist, ids, dm = run(path, d1, d2, th)
    assert dm.shape == (n1, n2)
    oracle_bits(dist, ids, d1, d2, th, dm)
    assert max_rel_err(dm, d1, d2) <= E_BOUND[path]
    Reference(d1, d2, E_BOUND[path]).check(ids, dist, th)
    return ids


@gpu
@pytest.mark.parametrize("n1", SIZES)
@pytest.mark.parametrize("path", list(PATHS))
def test_shapes(path, n1):
    for n2 in SIZES:
        ids = check_shape(path, n1, n2, 1000 * n1 + n2)
        if min(n1, n2) >= 63:
            assert len(ids) > 0


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_empty_key_split(path):
    """100 x 2049: the tensor-core path splits the keys 8 ways by 320, and the last split is empty"""
    check_shape(path, 100, 2049, 41)
    check_shape(path, 2049, 100, 42)


@gpu
@pytest.mark.parametrize("n1,n2", [(20000, 3000), (3000, 20000)])
@pytest.mark.parametrize("path", list(PATHS))
def test_one_split_regime(path, n1, n2):
    """more than 148 * 128 queries: one key split on that side, several on the other"""
    d1, d2 = correlated(n1, n2, 51)
    th = 0.99
    dist, ids, dm = run(path, d1, d2, th)
    assert max_rel_err(dm, d1, d2) <= E_BOUND[path]
    oracle_bits(dist, ids, d1, d2, th, dm)
    ref = Reference(d1, d2, E_BOUND[path], device=dev())
    _, _, pairs = ref.check(ids, dist, th)
    assert len(pairs) > 0.95 * min(n1, n2) // 2


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_65536_near_duplicates(path):
    """the ABI's largest sets: 64 blocks of 1024 rows in the single-CTA select kernel, no distance matrix"""
    n = 65536
    g = torch.Generator(device=dev()).manual_seed(61)
    d1 = torch.nn.functional.normalize(torch.randn(n, 128, device=dev(), generator=g), dim=1)
    d2 = d1[torch.randperm(n, device=dev(), generator=g)] + 0.03 * torch.randn(n, 128, device=dev(), generator=g)
    d2[: n // 4] = torch.randn(n // 4, 128, device=dev(), generator=g)      # a quarter without a partner
    d2 = torch.nn.functional.normalize(d2, dim=1)
    c = capi()
    c.debug_set(3, PATHS[path])
    try:
        dist, ids = c.match_smnn(d1, d2, 0.99)
    finally:
        c.debug_set(3, 0)
    ref = Reference(d1, d2, E_BOUND[path], device=dev())
    R, C, pairs = ref.check(ids.cpu().numpy(), dist.cpu().numpy()[:, 0], 0.99)
    assert len(ids) >= len(pairs) >= 0.7 * n
    # cross-check the GPU float64 summaries against NumPy on 512 sampled rows
    rows = np.random.default_rng(62).choice(n, 512, replace=False)
    D = sqdist64(d1[rows].cpu().numpy(), d2.cpu().numpy())
    np.testing.assert_allclose(np.sort(D, 1)[:, :2], ref.rows[0][rows].cpu().numpy(), rtol=0, atol=1e-12)
    assert np.array_equal(D.argmin(1), ref.rows[1][rows, 0].cpu().numpy())


@gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_non_unit_descriptors(path):
    d1, d2 = scaled_norms(*correlated(1500, 2049, 71), 72)
    for th in (1.0, 0.99):
        dist, ids, dm = run(path, d1, d2, th)
        assert max_rel_err(dm, d1, d2) <= E_BOUND[path]
        oracle_bits(dist, ids, d1, d2, th, dm)
        R, C, _ = Reference(d1, d2, E_BOUND[path]).check(ids, dist, th)
        assert float(torch.cat([R["determined"], C["determined"]]).float().mean()) >= 0.8


# ------------------------------------------------------------------------------------------ GPU: argument errors
def rejected(fn, exc, match):
    c = capi()
    torch.cuda.synchronize()
    before = c.launch_count()
    with pytest.raises(exc, match=match):
        fn()
    assert c.launch_count() == before


@gpu
def test_match_smnn_rejects_bad_descriptors():
    c = capi()
    a = torch.randn(10, 128, device=dev())
    rejected(lambda: c.match_smnn(a, a.cpu()), RuntimeError, "CUDA")
    rejected(lambda: c.match_smnn(a.cpu(), a), RuntimeError, "CUDA")
    rejected(lambda: c.match_smnn(a, a[:, :64].contiguous()), ValueError, r"\[n,128\]")
    rejected(lambda: c.match_smnn(a[:, :64].contiguous(), a), ValueError, r"\[n,128\]")
    rejected(lambda: c.match_smnn(a, torch.randn(10, 256, device=dev())), ValueError, r"\[n,128\]")
    rejected(lambda: c.match_smnn(a[None], a), ValueError, r"\[n,128\]")
    rejected(lambda: c.match_smnn(a, a.reshape(-1)), ValueError, r"\[n,128\]")
    rejected(lambda: c.match_smnn(a, a.int()), ValueError, "floating-point")
    if torch.cuda.device_count() > 1:
        rejected(lambda: c.match_smnn(a, a.to("cuda:1")), ValueError, "device")
    dist, ids = c.match_smnn(a, torch.zeros(0, device=dev()))      # an empty 1-D array is an empty set
    assert ids.shape == (0, 2)


@gpu
def test_c_abi_rejects_bad_match_arguments():
    c = capi()
    n = 65537
    a = torch.randn(n, 128, device=dev())
    ids = torch.zeros(n, 2, dtype=torch.int32, device=dev())
    dist = torch.zeros(n, device=dev())
    cnt = torch.zeros(1, dtype=torch.int32, device=dev())
    st = c._stream(dev())

    def call(n1, n2, dim, nbytes):
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev())
        return lambda: c._ok(c._match(c._ptr(a), n1, c._ptr(a), n2, dim, 0.99, c._ptr(ids), c._ptr(dist), c._ptr(cnt),
                                      None, c._ptr(ws), nbytes, st))

    big = int(c._match_ws(n, n))
    rejected(call(n, 100, 128, big), ValueError, "out of range")
    rejected(call(100, n, 128, big), ValueError, "out of range")
    rejected(call(-1, 100, 128, big), ValueError, "out of range")
    rejected(call(100, 100, 64, big), ValueError, "dimension")
    rejected(call(100, 100, 256, big), ValueError, "dimension")
    need = int(c._match_ws(1000, 2000))
    rejected(call(1000, 2000, 128, need - 1), ValueError, "workspace")
    rejected(call(1000, 2000, 128, 0), ValueError, "workspace")
    torch.cuda.synchronize()
    before = c.launch_count()
    call(1000, 2000, 128, need)()                                 # the same call with the workspace it asks for runs
    torch.cuda.synchronize()
    assert c.launch_count() > before


@gpu
def test_patch_and_hardnet_wrappers_reject_bad_arguments():
    c = capi()
    gray = torch.randint(0, 256, (2, 60, 80), dtype=torch.uint8, device=dev())
    kp = torch.rand(2, 5, 2, device=dev()) * 50 + 5
    cnt = torch.tensor([5, 3], dtype=torch.int32, device=dev())
    ok = c.extract_patches_batch(gray, kp, cnt, 10.0)
    rejected(lambda: c.extract_patches_batch(gray, kp.cpu(), cnt, 10.0), RuntimeError, "CUDA")
    rejected(lambda: c.extract_patches_batch(gray, kp, cnt.cpu(), 10.0), RuntimeError, "CUDA")
    rejected(lambda: c.extract_patches_batch(gray, kp[0], cnt, 10.0), ValueError, "keypoints")
    rejected(lambda: c.extract_patches_batch(gray, kp[:1], cnt, 10.0), ValueError, "keypoints")
    rejected(lambda: c.extract_patches_batch(gray, torch.cat([kp, kp[..., :1]], 2), cnt, 10.0), ValueError, "keypoints")
    rejected(lambda: c.extract_patches_batch(gray, kp, cnt[:1], 10.0), ValueError, "counts")
    rejected(lambda: c.extract_patches_batch(gray, kp, cnt[None], 10.0), ValueError, "counts")
    rejected(lambda: c.extract_patches_batch(gray, kp, cnt.float(), 10.0), ValueError, "counts")
    rejected(lambda: c.extract_patches_batch(gray[0], kp, cnt, 10.0), ValueError, "gray")
    if torch.cuda.device_count() > 1:
        rejected(lambda: c.extract_patches_batch(gray, kp.to("cuda:1"), cnt, 10.0), ValueError, "device")
    # an int64 count is converted, not reinterpreted
    assert torch.equal(c.extract_patches_batch(gray, kp, cnt.long(), 10.0), ok)
    assert torch.count_nonzero(ok[1, 3:]) == 0 and torch.count_nonzero(ok[1, :3]) > 0
    packed = torch.zeros(1, device=dev())
    for shape in ((4, 1, 16, 16), (4, 32, 32), (4, 2, 32, 32), (4, 1, 32, 64)):
        rejected(lambda: c.hardnet_forward(torch.rand(*shape, device=dev()), packed), ValueError, "32,32")
