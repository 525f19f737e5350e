"""ORACLE-side synthetic input generators (test infrastructure only): seeded stick-figure heat/PAF maps in the
reference's 19-heat / 38-PAF COCO layout (SURVEY.md appendix B), and noise maps.  These are INPUTS for parity
tests, not a restatement of any reference function."""
import numpy as np

LIMB_PARTS = [(1, 2), (1, 5), (2, 3), (3, 4), (5, 6), (6, 7), (1, 8), (8, 9), (9, 10), (1, 11), (11, 12), (12, 13),
              (1, 0), (0, 14), (14, 16), (0, 15), (15, 17), (2, 16), (5, 17)]
LIMB_PAF_CH = [(12, 13), (20, 21), (14, 15), (16, 17), (22, 23), (24, 25), (0, 1), (2, 3), (4, 5), (6, 7), (8, 9),
               (10, 11), (28, 29), (30, 31), (34, 35), (32, 33), (36, 37), (18, 19), (26, 27)]
# canonical skeleton in a unit box (x, y), 18 COCO parts
_SKEL = np.array([[.50, .08], [.50, .22], [.36, .22], [.30, .40], [.27, .56], [.64, .22], [.70, .40], [.73, .56],
                  [.42, .55], [.41, .75], [.40, .95], [.58, .55], [.59, .75], [.60, .95], [.46, .05], [.54, .05],
                  [.41, .07], [.59, .07]])


def stick_figures(num_persons, seed, h=46, w=46, stride=8, sigma=7.0, paf_width=6.0, drop_prob=0.1):
    """Returns (heat [h,w,19] float32, paf [h,w,38] float32, keypoints [P,18,3] (x,y,visible) in image pixels)."""
    rs = np.random.RandomState(seed)
    H, W = h * stride, w * stride
    heat = np.zeros((h, w, 19), np.float32)
    paf = np.zeros((h, w, 38), np.float32)
    cnt = np.zeros((h, w, 19), np.float32)
    ys, xs = np.mgrid[0:h, 0:w]
    cx = xs * stride + stride / 2.0 - 0.5
    cy = ys * stride + stride / 2.0 - 0.5
    kps = np.zeros((num_persons, 18, 3))
    for p in range(num_persons):
        size = rs.uniform(0.28, 0.6) * min(H, W)
        ox = rs.uniform(0, W - size * 0.5)
        oy = rs.uniform(0, H - size)
        ang = rs.uniform(-0.35, 0.35)
        rot = np.array([[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]])
        pts = (_SKEL - 0.5) @ rot.T * size + [ox + size * 0.5, oy + size * 0.5] + rs.normal(0, size * 0.015, (18, 2))
        vis = (rs.rand(18) > drop_prob) & (pts[:, 0] >= 0) & (pts[:, 0] < W) & (pts[:, 1] >= 0) & (pts[:, 1] < H)
        kps[p, :, :2] = pts
        kps[p, :, 2] = vis
        for j in range(18):
            if not vis[j]:
                continue
            g = np.exp(-((cx - pts[j, 0]) ** 2 + (cy - pts[j, 1]) ** 2) / (2 * sigma * sigma))
            heat[:, :, j] = np.maximum(heat[:, :, j], g * rs.uniform(0.75, 1.0))
        for l, (a, b) in enumerate(LIMB_PARTS):
            if not (vis[a] and vis[b]):
                continue
            v = pts[b] - pts[a]
            n = np.linalg.norm(v)
            if n < 1e-3:
                continue
            u = v / n
            rx, ry = cx - pts[a, 0], cy - pts[a, 1]
            along = rx * u[0] + ry * u[1]
            perp = np.abs(rx * u[1] - ry * u[0])
            m = (along >= 0) & (along <= n) & (perp <= paf_width)
            paf[:, :, LIMB_PAF_CH[l][0]][m] += u[0]
            paf[:, :, LIMB_PAF_CH[l][1]][m] += u[1]
            cnt[:, :, l][m] += 1
    for l in range(19):
        m = cnt[:, :, l] > 1
        for ch in LIMB_PAF_CH[l]:
            paf[:, :, ch][m] /= cnt[:, :, l][m]
    heat[:, :, 18] = 1.0 - heat[:, :, :18].max(axis=2)
    heat += rs.normal(0, 0.004, heat.shape).astype(np.float32)   # breaks exact ties / plateaus
    paf += rs.normal(0, 0.004, paf.shape).astype(np.float32)
    return heat.astype(np.float32), paf.astype(np.float32), kps


def noise_maps(seed, h=46, w=46, heat_scale=0.45, paf_scale=0.6):
    """Maps with the statistics of a random-weight network (thousands of peaks): the stress case."""
    rs = np.random.RandomState(seed)
    heat = (rs.standard_normal((h, w, 19)) * heat_scale).astype(np.float32)
    paf = (rs.standard_normal((h, w, 38)) * paf_scale).astype(np.float32)
    return heat, paf


# ---------------------------------------------------------------------------------------------------------------
# Fuzz scenarios for the pafprocess stage (joint list + low-resolution PAF maps, no NMS involved): used to compare the
# reference's compiled pafprocess.cpp with the product's cores on inputs the stick-figure fixtures do not reach
# (cross links between persons, duplicated peaks on one pixel, exact score ties, masked fields).
_LIMBS = [(1, 2), (1, 5), (2, 3), (3, 4), (5, 6), (6, 7), (1, 8), (8, 9), (9, 10), (1, 11), (11, 12), (12, 13), (1, 0),
          (0, 14), (14, 16), (0, 15), (15, 17), (2, 16), (5, 17)]                       # pafprocess.h:21-24
_PAFCH = [(12, 13), (20, 21), (14, 15), (16, 17), (22, 23), (24, 25), (0, 1), (2, 3), (4, 5), (6, 7), (8, 9), (10, 11),
          (28, 29), (30, 31), (34, 35), (32, 33), (36, 37), (18, 19), (26, 27)]           # pafprocess.h:16-19


def fuzz_field(rs, h, w, kind):
    """Random peaks (kind: 'uniform' | 'cluster' | 'ties') + per-limb (nearly) constant direction fields."""
    maxp = int(rs.choice([1, 2, 3, 5, 8]))
    rows = []
    centers = rs.randint(8, min(h, w) * 8 - 8, (int(rs.randint(1, 6)), 2))
    for part in range(18):
        for _ in range(int(rs.randint(0, maxp + 1))):
            if kind in ("cluster", "ties") and rs.rand() < 0.8:
                c = centers[rs.randint(len(centers))]
                spread = 3 if kind == "ties" else 40
                x = int(np.clip(c[0] + rs.randint(-spread, spread + 1), 0, w * 8 - 1))
                y = int(np.clip(c[1] + rs.randint(-spread, spread + 1), 0, h * 8 - 1))
            else:
                x, y = int(rs.randint(0, w * 8)), int(rs.randint(0, h * 8))
            rows.append((x, y, float(np.float32(rs.choice([0.2, 0.5, 0.9, rs.rand()]))), 0, part))
    jl = np.array(rows, np.float32).reshape(-1, 5)
    jl[:, 3] = np.arange(len(jl))
    paf = np.zeros((h, w, 38), np.float32)
    for ch in range(0, 38, 2):
        ang = rs.choice([0, np.pi / 2, np.pi, 3 * np.pi / 2, np.pi / 4]) if kind == "ties" else rs.rand() * 2 * np.pi
        mag = rs.choice([0.3, 0.6, 1.0])
        noise = 0.0 if kind == "ties" else 0.3
        paf[:, :, ch] = np.cos(ang) * mag + noise * rs.randn(h, w)
        paf[:, :, ch + 1] = np.sin(ang) * mag + noise * rs.randn(h, w)
        if rs.rand() < 0.3:
            paf[:, :, ch:ch + 2] *= (rs.rand(h, w, 1) < 0.7)
    return jl, np.ascontiguousarray(paf.astype(np.float32))


def fuzz_persons(rs, h, w):
    """1-6 loosely person-shaped peak sets with their true limbs drawn into the PAF maps, random cross links between
    persons (ambiguous assignments, merges of partial persons) and duplicated peaks (exact score ties)."""
    K = int(rs.randint(1, 7))
    pts = {}
    for k in range(K):
        c = rs.randint(40, min(h, w) * 8 - 40, 2)
        sc = rs.randint(10, 45)
        for part in range(18):
            if rs.rand() < 0.85:
                pts[(k, part)] = (int(np.clip(c[0] + rs.randint(-sc, sc + 1), 0, w * 8 - 1)),
                                  int(np.clip(c[1] + rs.randint(-sc, sc + 1), 0, h * 8 - 1)))
    rows = []
    for part in range(18):
        for k in range(K):
            if (k, part) in pts:
                x, y = pts[(k, part)]
                rows.append((x, y, float(np.float32(rs.choice([0.3, 0.6, 0.95]))), 0, part))
                if rs.rand() < 0.15:
                    rows.append((x + int(rs.randint(0, 2)), y, float(np.float32(0.6)), 0, part))
    jl = np.array(rows, np.float32).reshape(-1, 5)
    jl[:, 3] = np.arange(len(jl))
    paf = np.zeros((h, w, 38), np.float32)

    def draw(a, b, chx, chy, mag):
        ax, ay, bx, by = a[0] / 8.0, a[1] / 8.0, b[0] / 8.0, b[1] / 8.0
        d = np.array([bx - ax, by - ay])
        nrm = np.linalg.norm(d)
        if nrm < 1e-6:
            return
        u = d / nrm
        for t in np.linspace(0, 1, int(nrm * 2) + 2):
            px, py = ax + t * d[0], ay + t * d[1]
            for ox in (-1, 0, 1):
                for oy in (-1, 0, 1):
                    xi, yi = int(round(px)) + ox, int(round(py)) + oy
                    if 0 <= xi < w and 0 <= yi < h:
                        paf[yi, xi, chx] = u[0] * mag
                        paf[yi, xi, chy] = u[1] * mag
    for l, (pa, pb) in enumerate(_LIMBS):
        for k in range(K):
            if (k, pa) in pts and (k, pb) in pts and rs.rand() < 0.9:
                draw(pts[(k, pa)], pts[(k, pb)], _PAFCH[l][0], _PAFCH[l][1], float(rs.choice([0.5, 0.8, 1.0])))
            k2 = int(rs.randint(K))
            if k2 != k and (k, pa) in pts and (k2, pb) in pts and rs.rand() < 0.35:
                draw(pts[(k, pa)], pts[(k2, pb)], _PAFCH[l][0], _PAFCH[l][1], float(rs.choice([0.5, 0.8, 1.0])))
    return jl, np.ascontiguousarray(paf)


def fuzz_scenario(t):
    """Scenario t of the pafprocess fuzz tests: (h, w, joint list, paf [h,w,38]); odd t person-shaped, even t random
    fields (uniform / cluster / ties in turn)."""
    rs = np.random.RandomState(1000 + t)
    h, w = int(rs.choice([12, 23, 46])), int(rs.choice([23, 46, 53]))
    if t % 2:
        h = max(h, 23)
        jl, paf = fuzz_persons(rs, h, w)
    else:
        jl, paf = fuzz_field(rs, h, w, ("uniform", "cluster", "ties")[(t // 2) % 3])
    return h, w, jl, paf
