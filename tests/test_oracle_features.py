"""The LOAM front-end oracle (oracle/feature_oracle.cpp) against a plain-Python loop restatement of the contract, on small scans
built to reach every quirk listed in its header.  The restatement also counts the events each scan reaches, so that a scan that
stops reaching a quirk fails here."""
import math

import numpy as np
import pytest

import feature_scans

F = np.float32


@pytest.fixture(scope="module")
def oracle():
    from oracle import feature_binding
    feature_binding.build()
    return feature_binding


def voxel_grid(xyzi, leaf):
    """pcl::VoxelGrid (min points 0) with pcl::CentroidPoint's arithmetic: fp32 sums in input order, divided by the count."""
    p = np.asarray(xyzi, F)
    inv = F(1.0) / F(leaf)
    min_b = np.floor(p[:, :3].min(0) * inv).astype(np.int64)
    div_b = np.floor(p[:, :3].max(0) * inv).astype(np.int64) - min_b + 1
    ijk = (np.floor(p[:, :3] * inv) - min_b.astype(F)).astype(np.int64)
    idx = ijk[:, 0] + ijk[:, 1] * div_b[0] + ijk[:, 2] * div_b[0] * div_b[1]
    out = []
    for key in sorted(set(idx.tolist())):
        s = np.zeros(4, F)
        members = np.flatnonzero(idx == key)
        for k in members:
            s = s + p[k]
        out.append(s / F(len(members)))
    return np.array(out, F).reshape(-1, 4)


def restate(rec, stride, int_off, ring_off, ring_bytes, prm):
    """The contract, one loop per step, fp32 through numpy scalars.  Returns (outputs, events)."""
    N, H = prm.n_scan, prm.horizon_scan
    ev = dict(nonfinite=0, range=0, row=0, col=0, dup=0, corner21=0, surf_blocks_next_corner=0, ep_picked=0, index4=0, walk_below_zero=0,
              corner_tie=0, zero_tie=0, leading_empty=0, short_ring=0, livox_past_h=0, walk_gap_stop=0)
    n = len(rec)
    owner, rmat, cnt = {}, {}, [0] * N
    ang = F(360.0 / float(F(H)))
    for i in range(n):
        x, y, z = (float(v) for v in rec[i, 0:12].view(F))
        if not (math.isfinite(x) and math.isfinite(y) and math.isfinite(z)):
            ev["nonfinite"] += 1
            continue
        x, y, z = F(x), F(y), F(z)
        rng = np.sqrt((x * x + y * y) + z * z)
        if rng < F(prm.min_range) or rng > F(prm.max_range):
            ev["range"] += 1
            continue
        row = int(rec[i, ring_off]) | ((int(rec[i, ring_off + 1]) << 8) if ring_bytes == 2 else 0)
        if row >= N or row % prm.downsample_rate != 0:
            ev["row"] += 1
            continue
        if prm.sensor == 1:
            c = cnt[row]
            cnt[row] += 1
        else:
            a = F(math.atan2(float(x), float(y)))
            ha = F(float(a * F(180.0)) / math.pi)
            q = (float(ha) - 90.0) / float(ang)
            rq = math.floor(abs(q) + 0.5) * (1 if q >= 0 else -1)
            c = int(-rq + H // 2)
            if c >= H:
                c -= H
        if c < 0 or c >= H:
            ev["col"] += 1
            ev["livox_past_h"] += prm.sensor == 1
            continue
        if (row, c) in owner:
            ev["dup"] += 1
            continue
        owner[(row, c)] = i
        rmat[(row, c)] = rng
    cloud, col, r, S, E = [], [], [], [], []
    for i in range(N):
        S.append(len(r) - 1 + 5)
        for j in range(H):
            if (i, j) in owner:
                o = owner[(i, j)]
                v = rec[o, 0:12].view(F)
                cloud.append([v[0], v[1], v[2], rec[o, int_off:int_off + 4].view(F)[0]])
                col.append(j)
                r.append(rmat[(i, j)])
        E.append(len(r) - 1 - 5)
        ev["leading_empty"] += S[-1] - 4 == E[-1] + 6 == 0
        ev["short_ring"] += 0 < (E[-1] + 6) - (S[-1] - 4) < 11
    m = len(r)
    curv = [F(0)] * m
    picked, label = [0] * m, [0] * m
    ent = [(F(0), i) for i in range(m)]
    for i in range(5, m - 5):
        d = r[i - 5]
        for k in (-4, -3, -2, -1):
            d = d + r[i + k]
        d = d - r[i] * F(10)
        for k in (1, 2, 3, 4, 5):
            d = d + r[i + k]
        curv[i] = d * d
        ent[i] = (curv[i], i)
    for i in range(5, m - 6):
        if abs(col[i + 1] - col[i]) < 10:
            if float(r[i] - r[i + 1]) > 0.3:
                for k in range(6):
                    picked[i - k] = 1
            elif float(r[i + 1] - r[i]) > 0.3:
                for k in range(1, 7):
                    picked[i + k] = 1
        if float(abs(r[i - 1] - r[i])) > 0.02 * float(r[i]) and float(abs(r[i + 1] - r[i])) > 0.02 * float(r[i]):
            picked[i] = 1
    marker = {}

    def mark(ind, who, lo_hi):
        picked[ind] = 1
        marker[ind] = who
        lo_hi[0], lo_hi[1] = min(lo_hi[0], ind), max(lo_hi[1], ind)
        for l in range(1, 6):
            if abs(col[ind + l] - col[ind + l - 1]) > 10:
                ev["walk_gap_stop"] += 1
                break
            picked[ind + l] = 1
            marker[ind + l] = who
            lo_hi[1] = max(lo_hi[1], ind + l)
        for l in range(-1, -6, -1):
            if ind + l < 0:
                ev["walk_below_zero"] += 1
                break
            if abs(col[ind + l] - col[ind + l + 1]) > 10:
                ev["walk_gap_stop"] += 1
                break
            picked[ind + l] = 1
            marker[ind + l] = who
            lo_hi[0] = min(lo_hi[0], ind + l)

    corner, surface = [], []
    for i in range(N):
        rs = []
        lo_hi = [1 << 60, -(1 << 60)]
        for j in range(6):
            sp = int((S[i] * (6 - j) + E[i] * j) / 6)
            ep = int((S[i] * (5 - j) + E[i] * (j + 1)) / 6) - 1
            if sp >= ep:
                continue
            ev["index4"] += sp == 4
            ent[sp:ep] = sorted(ent[sp:ep])
            ev["zero_tie"] += sum(ent[k][0] == ent[k + 1][0] == 0 for k in range(sp, ep - 1))
            largest = 0
            for k in range(ep, sp - 1, -1):
                ind = ent[k][1]
                if picked[ind] and curv[ind] > F(prm.edge_threshold) and marker.get(ind) == (i, j - 1, "surf"):
                    ev["surf_blocks_next_corner"] += 1
                if picked[ind] == 0 and curv[ind] > F(prm.edge_threshold):
                    largest += 1
                    if largest > 20:
                        ev["corner21"] += 1
                        break
                    ev["corner_tie"] += k > sp and ent[k - 1][0] == ent[k][0]
                    label[ind] = 1
                    corner.append(cloud[ind])
                    mark(ind, (i, j, "corner"), lo_hi)
            for k in range(sp, ep + 1):
                ind = ent[k][1]
                if picked[ind] == 0 and curv[ind] < F(prm.surf_threshold):
                    label[ind] = -1
                    mark(ind, (i, j, "surf"), lo_hi)
            ev["ep_picked"] += label[ep] != 0
            for k in range(sp, ep + 1):
                if label[k] <= 0:
                    rs.append(cloud[k])
        if lo_hi[1] >= lo_hi[0]:  # quirk 6: step-5 marks of ring i stay within [S_i - 5, E_i + 4]
            assert S[i] - 5 <= lo_hi[0] and lo_hi[1] <= E[i] + 4, (i, lo_hi, S[i], E[i])
        if rs:
            surface.extend(voxel_grid(np.array(rs, F), prm.odometry_surf_leaf))
    corner = np.array(corner, F).reshape(-1, 4)
    surface = np.array(surface, F).reshape(-1, 4)
    out = dict(cloud=np.array(cloud, F).reshape(-1, 4), col=np.array(col, np.int32), range=np.array(r, F), start=np.array(S, np.int32),
               end=np.array(E, np.int32), curvature=np.array(curv, F), label=np.array(label, np.int8), picked=np.array(picked, np.uint8),
               corner=corner, surface=surface)
    out["corner_ds"] = voxel_grid(corner, prm.mapping_corner_leaf) if len(corner) else np.zeros((0, 4), F)
    out["surf_ds"] = voxel_grid(surface, prm.mapping_surf_leaf) if len(surface) else np.zeros((0, 4), F)
    return out, ev


def _compare(oracle, scan):
    rec, stride, io, ro, rb, prm = scan
    got = oracle.features(rec, stride, io, ro, rb, prm)
    want, ev = restate(rec.reshape(-1, stride), stride, io, ro, rb, prm)
    for k in ("cloud", "col", "range", "start", "end", "curvature", "label", "picked", "corner", "surface", "corner_ds", "surf_ds"):
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), k
    assert (got["dropped_nonfinite"], got["dropped_range"], got["dropped_row"], got["dropped_col"], got["dropped_dup"]) == (
        ev["nonfinite"], ev["range"], ev["row"], ev["col"], ev["dup"])
    return got, ev


def test_quirk_scan_matches_restatement(oracle):
    got, ev = _compare(oracle, feature_scans.quirks())
    for k in ("corner21", "ep_picked", "index4", "walk_below_zero", "corner_tie", "zero_tie", "leading_empty", "short_ring", "livox_past_h"):
        assert ev[k] > 0, k
    assert got["n_corner"] > 0 and got["n_surface"] > 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_spinning_scan_matches_restatement(oracle, seed):
    got, ev = _compare(oracle, feature_scans.spinning(n_scan=8, H=240, seed=seed, dup=0.2, junk=0.05))
    for k in ("dup", "nonfinite", "range", "row"):
        assert ev[k] > 0, k
    assert got["n_corner_ds"] > 0 and got["n_surf_ds"] > 0


def test_surf_pick_blocks_next_region_corner(oracle):
    _, ev = _compare(oracle, feature_scans.spinning(n_scan=8, H=360, seed=0))
    assert ev["surf_blocks_next_corner"] > 0 and ev["walk_gap_stop"] > 0


def test_downsample_rate_and_livox(oracle):
    _compare(oracle, feature_scans.spinning(n_scan=8, H=240, seed=4, rate=2))
    got, ev = _compare(oracle, feature_scans.livox())
    assert ev["livox_past_h"] > 0 and got["n_corner"] > 0


def test_empty_and_tiny_scans(oracle):
    rec, stride, io, ro, rb, prm = feature_scans.spinning(n_scan=4, H=120, seed=5)
    for k in (0, 1, 5, 11, 12):
        got, _ = _compare(oracle, (rec[:k], stride, io, ro, rb, prm))
        assert got["n_extracted"] <= k
