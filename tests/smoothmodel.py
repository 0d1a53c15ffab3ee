"""Independent pure-Python model of the smoothing specification (DESIGN.md section 5), small cases only.

Written from the prose of DESIGN.md section 5, not from oracle/tmc2_oracle.c: plain loops over the points and Python
integers throughout, so no quantity has a width.  Its input is what rows a-1 to a-9 already pin (the pre-smoothing
positions and colours, the partition and the boundary types of a frame); its output is the smoothed frame, the moved and
recoloured counts and, for every type-1 point that reaches a comparison, the exact two sides of that comparison:

  geometry          lhs = 2*count*|d|^2 + 65536          against rhs = 262144*max(threshold, count)   (moves when lhs >= rhs)
  colour, per cell  num = cnt*sum(Y^2) - sum(Y)^2         against lim = (t_var*cnt)^2                  (unusable when num > lim)
                    dy  = |meanY_q8 - 256*Y|              against 256*t_diff                           (unusable when dy > it)
  colour, per point dist = 10|dY| + |dU| + |dV|           against t_smooth                             (recoloured when dist >= t_smooth, dist > 0)

Test infrastructure only.
"""


class Unsupported(Exception):
    """The grid is wider than 1024 cells (the specification refuses it)."""


class Grid:
    def __init__(self, g, bitdepth):
        self.g = g
        self.w = -(-(1 << bitdepth) // g)
        if self.w > 1024:
            raise Unsupported(f"grid of edge {g} at bit depth {bitdepth} is {self.w} cells wide")
        self.th = g * self.w
        self.disth = max(g // 2, 1)

    def cell(self, p):
        """Cell of a point, or None when a coordinate is >= th."""
        if any(c >= self.th for c in p):
            return None
        return tuple(c // self.g for c in p)

    def inside_margin(self, p):
        return all(c >= self.disth and c + self.disth < self.th for c in p)

    def neighbourhood(self, p):
        """The 2x2x2 cells around p with their trilinear weights over (2g)^3: [(cell or None, weight)]."""
        g = self.g
        lo, wa = [], []
        for c in p:
            s = c // g - (1 if c % g < g // 2 else 0)
            lo.append(s)
            wa.append(2 * (c - s * g - g // 2) + 1)
        out = []
        for dz in (0, 1):
            for dy in (0, 1):
                for dx in (0, 1):
                    d = (dx, dy, dz)
                    cell = tuple(lo[a] + d[a] for a in range(3))
                    wgt = 1
                    for a in range(3):
                        wgt *= wa[a] if d[a] else 2 * g - wa[a]
                    ok = all(0 <= c < self.w for c in cell)
                    out.append((cell if ok else None, wgt))
        return out


def q8_mean(s, n):
    return (256 * s + n // 2) // n


def round_q8(c4):
    return min((c4 + 128) >> 8, 65535)


def threshold_scale(attribute_bitdepth):
    return 1 << (attribute_bitdepth - 8) if attribute_bitdepth > 8 else 1


def _stats(points, grid):
    """Per cell: count, sums of the given per-point vectors, patch indices seen.  points: (position, patch, vector)."""
    cells = {}
    for p, part, vec in points:
        c = grid.cell(p)
        if c is None:
            continue
        e = cells.setdefault(c, {"count": 0, "sums": None, "patches": set()})
        e["count"] += 1
        e["sums"] = list(vec) if e["sums"] is None else [a + b for a, b in zip(e["sums"], vec)]
        e["patches"].add(part)
    return cells


def _merge(cells, prior, g=None):
    """Add leftover cell statistics (cell_statistics) into `cells`.  A leftover cell lands on the cell with the same
    coordinates (the key of a hashed table, and the dense index cx + w*(cy + w*cz) when the slot count is the same); its
    patch set joins the cell's, because its claim word still holds `patch + 1`.  Geometry sums are kept relative to the cell
    origin (as the tables hold them), so they are re-based on this grid's origin of that cell (`g`)."""
    for c, (cnt, sums, patches) in prior.items():
        if g is not None:
            sums = [s + cnt * c[a] * g for a, s in enumerate(sums)]
        e = cells.setdefault(c, {"count": 0, "sums": [0] * len(sums), "patches": set()})
        e["count"] += cnt
        e["sums"] = [a + b for a, b in zip(e["sums"], sums)]
        e["patches"] |= set(patches)


def cell_statistics(params, positions, colors, partition, btype):
    """What one frame leaves in the cell tables when nothing clears them: {"geo": {cell: (count, sums relative to the cell
    origin, patches)}, "col": {cell: (count, [sum Y, sum U, sum V, sum Y^2], patches)}}.  The patch identity is the index of
    the patch within its frame (what the claim word holds, minus one)."""
    pos = [tuple(int(c) for c in p) for p in positions]
    part = [int(x) for x in partition]
    bt = [int(x) for x in btype]
    out = {"geo": {}, "col": {}}
    if params.geometry_smoothing:
        G = Grid(params.grid_size, params.geometry_bitdepth_3d)
        for c, e in _stats([(pos[k], part[k], pos[k]) for k in range(len(pos))], G).items():
            out["geo"][c] = (e["count"], [s - e["count"] * c[a] * G.g for a, s in enumerate(e["sums"])], e["patches"])
    if params.color_smoothing and colors is not None and params.attribute_count:
        G = Grid(params.cgrid_size, params.geometry_bitdepth_3d)
        col = [tuple(int(c) for c in x) for x in colors]
        pts = [(pos[k], part[k], (col[k][0], col[k][1], col[k][2], col[k][0] ** 2)) for k in range(len(pos)) if bt[k] == 2]
        out["col"] = {c: (e["count"], e["sums"], e["patches"]) for c, e in _stats(pts, G).items()}
    return out


def smooth(params, positions, colors, partition, btype, prior=None):
    """positions / colors: sequences of 3 ints per point (colors may be None), partition / btype: one int per point.
    prior: leftover cell statistics of an earlier frame (cell_statistics), merged into the cells before the filters run --
    the tables of a launch whose cells were not cleared.

    Returns dict(positions, colors, moved, recoloured, geo, col, type2_per_cell) where geo / col map the point index of
    every type-1 point that reached a comparison to its quantities."""
    n = len(positions)
    pos = [tuple(int(c) for c in p) for p in positions]
    col = None if colors is None else [tuple(int(c) for c in x) for x in colors]
    part = [int(x) for x in partition]
    bt = [int(x) for x in btype]
    out_pos, out_col = list(pos), None if col is None else list(col)
    moved = recoloured = 0
    geo_log, col_log, type2 = {}, {}, {}

    if params.geometry_smoothing:
        G = Grid(params.grid_size, params.geometry_bitdepth_3d)
        cells = _stats([(pos[k], part[k], pos[k]) for k in range(n)], G)
        if prior:
            _merge(cells, prior.get("geo", {}), G.g)
        thr = params.threshold_smoothing
        for k in range(n):
            p = pos[k]
            if bt[k] != 1 or G.cell(p) is None or not G.inside_margin(p):
                continue
            nb = G.neighbourhood(p)
            used = [(cells.get(c) if c is not None else None, w) for c, w in nb]
            if not any(e is not None and len(e["patches"]) > 1 for e, _ in used):
                continue
            w3 = (2 * G.g) ** 3
            cnt_w = sum(w * e["count"] for e, w in used if e is not None)
            count = cnt_w // w3
            if count == 0:
                continue
            c4 = []
            for a in range(3):
                acc = sum(w * (q8_mean(e["sums"][a], e["count"]) if e is not None else 256 * p[a]) for e, w in used)
                c4.append((acc + w3 // 2) // w3)
            d2 = sum((256 * p[a] - c4[a]) ** 2 for a in range(3))
            lhs = 2 * count * d2 + 65536
            rhs = 262144 * max(thr, count)
            geo_log[k] = dict(lhs=lhs, rhs=rhs, count=count, d2=d2)
            if lhs >= rhs:
                q = tuple(round_q8(c) for c in c4)
                if q != p:
                    moved += 1
                out_pos[k] = q

    if params.color_smoothing and col is not None and params.attribute_count:
        G = Grid(params.cgrid_size, params.geometry_bitdepth_3d)
        sc = threshold_scale(params.attribute_bitdepth)
        t_smooth = params.threshold_color_smoothing * sc
        t_diff = params.threshold_color_difference * sc
        t_var = params.threshold_color_variation * sc
        pts = [(pos[k], part[k], (col[k][0], col[k][1], col[k][2], col[k][0] ** 2)) for k in range(n) if bt[k] == 2]
        cells = _stats(pts, G)
        if prior:
            _merge(cells, prior.get("col", {}))
        for c, e in cells.items():
            type2[c] = e["count"]
        for k in range(n):
            p, y = pos[k], col[k]
            if bt[k] != 1 or G.cell(p) is None or not G.inside_margin(p):
                continue
            nb = G.neighbourhood(p)
            used = [(cells.get(c) if c is not None else None, w) for c, w in nb]
            if not any(e is not None and len(e["patches"]) > 1 for e, _ in used):
                continue
            w3 = (2 * G.g) ** 3
            acc = [0, 0, 0]
            log = dict(var=[], diff=[])
            for e, w in used:
                src = [256 * v for v in y]
                if e is not None:
                    cnt, (sy, su, sv, sy2) = e["count"], e["sums"]
                    mean = [q8_mean(s, cnt) for s in (sy, su, sv)]
                    num, lim = cnt * sy2 - sy * sy, (t_var * cnt) ** 2
                    dy = abs(mean[0] - 256 * y[0])
                    log["var"].append((num, lim))
                    log["diff"].append((dy, 256 * t_diff))
                    if num <= lim and dy <= 256 * t_diff:
                        src = mean
                for a in range(3):
                    acc[a] += w * src[a]
            q = tuple(round_q8((acc[a] + w3 // 2) // w3) for a in range(3))
            dist = 10 * abs(q[0] - y[0]) + abs(q[1] - y[1]) + abs(q[2] - y[2])
            log["dist"] = (dist, t_smooth)
            col_log[k] = log
            if dist >= t_smooth and dist > 0:
                out_col[k] = q
                recoloured += 1

    return dict(positions=out_pos, colors=out_col, moved=moved, recoloured=recoloured, geo=geo_log, col=col_log,
                type2_per_cell=type2)


def _presmooth(frame):
    colors = frame["colors16bit_presmooth"] if frame["with_colors"] and len(frame["colors16bit_presmooth"]) else None
    if colors is None and frame["with_colors"]:
        colors = frame["colors16bit"]
    return (frame["positions_presmooth"].tolist(), None if colors is None else colors.tolist(), frame["partition"].tolist(),
            frame["boundary_type"].tolist())


def smooth_oracle_frame(params, frame, prior=None):
    """smooth() on the pre-smoothing streams of an oracle frame (oracle.reconstruct_frame)."""
    return smooth(params, *_presmooth(frame), prior=prior)


def oracle_frame_statistics(params, frame):
    """cell_statistics() of an oracle frame, under `params` (the grids of the launch that left them)."""
    return cell_statistics(params, *_presmooth(frame))
