"""numpy port of the brute-force nearest-point loop of the reference's SDF caller (src/sdf_field.cpp:212-249) and of its
border-distance rows, the reference the tests of fi_nearest_point_distance and fi_field_add_border_distance compare
against bit for bit.  Every operation is a float32 numpy ufunc, so each product and sum rounds on its own (no FMA).

    dx_d = p_i[d] - q[d];  d2_i = dx_0 * dx_0 + dx_1 * dx_1 (+ dx_2 * dx_2)
    closest = min over i of d2_i, NaN skipped (std::min(closest, d2_i));  distance = sqrt(closest)
    nearest = the first i with d2_i == closest, -1 when closest is +inf

Also a chunked torch brute force of the same loop for the GPU tests (large clouds)."""
import numpy as np

F = np.float32


def d2_row(points, q):
    """fp32 d2 of every point to one query, left to right over the axes."""
    p = np.asarray(points, F)
    q = np.asarray(q, F)
    dx = (p[:, 0] - q[0]).astype(F)
    d2 = (dx * dx).astype(F)
    for d in range(1, p.shape[1]):
        dd = (p[:, d] - q[d]).astype(F)
        d2 = (d2 + (dd * dd).astype(F)).astype(F)
    return d2


def nearest(points, queries):
    """(distances float32 (m,), nearest int64 (m,)) of the loop."""
    queries = np.asarray(queries, F)
    points = np.asarray(points, F).reshape(-1, queries.shape[1])
    m = queries.shape[0]
    dist, idx = np.full(m, np.inf, F), np.full(m, -1, np.int64)
    if points.shape[0] == 0:
        return dist, idx
    with np.errstate(all="ignore"):
        for j in range(m):
            d2 = d2_row(points, queries[j])
            d2 = np.where(np.isnan(d2), F(np.inf), d2)
            c = d2.min()
            dist[j] = np.sqrt(c)
            if c < np.inf:
                idx[j] = int(np.argmax(d2 == c))
    return dist, idx


def border_nodes(sizes):
    """Linear indices of the border nodes in ascending order (x fastest)."""
    sizes = list(sizes)
    coords = np.indices(sizes[::-1]).reshape(len(sizes), -1)[::-1]  # coords[d] of every node in linear order
    on = np.zeros(coords.shape[1], bool)
    for d, n in enumerate(sizes):
        on |= (coords[d] == 0) | (coords[d] == n - 1)
    return np.nonzero(on)[0].astype(np.int64), coords[:, on].T.astype(F)


def border_rows(sizes, weight, positions):
    """The rows the caller's loop appends with add_equation: (cols int32, vals float32, rhs float32), one triplet each;
    nothing when weight == 0."""
    w = F(weight)
    if w == 0:
        return np.zeros(0, np.int32), np.zeros(0, F), np.zeros(0, F)
    nodes, q = border_nodes(sizes)
    dist, _ = nearest(np.asarray(positions, F).reshape(-1, len(sizes)), q)
    with np.errstate(all="ignore"):
        return nodes.astype(np.int32), np.full(nodes.size, F(1.0) * w, F), (dist * w).astype(F)


def torch_nearest(points, queries, chunk=None):
    """The loop on the GPU by brute force: separate elementwise ops (never cdist, whose matrix product is not
    bit-exact), NaN d2 mapped to +inf before the minimum, chunks of points merged in ascending order replacing only on
    a strict <.  points (n, D) and queries (m, D) are float32 CUDA tensors; chunks of about 2^28 pairs by default.
    Its cost is exactly linear in the number of queries.  Returns (distances, nearest)."""
    import torch
    m, D = queries.shape
    chunk = chunk or max(256, (1 << 28) // max(m, 1))
    best = torch.full((m,), float("inf"), dtype=torch.float32, device=queries.device)
    bi = torch.full((m,), -1, dtype=torch.int64, device=queries.device)
    for a in range(0, points.shape[0], chunk):
        p = points[a:a + chunk]
        dx = p[None, :, 0] - queries[:, None, 0]
        d2 = dx * dx
        for d in range(1, D):
            dd = p[None, :, d] - queries[:, None, d]
            d2 = d2 + dd * dd
        d2 = torch.where(torch.isnan(d2), torch.full_like(d2, float("inf")), d2)
        c, k = torch.min(d2, dim=1)  # first index of the minimum within the chunk
        better = c < best
        best = torch.where(better, c, best)
        bi = torch.where(better, k + a, bi)
    bi = torch.where(best < float("inf"), bi, torch.full_like(bi, -1))
    return torch.sqrt(best), bi
