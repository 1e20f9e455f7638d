"""TEST INFRASTRUCTURE (oracle) -- float64 numpy restatements of the contracts of single C-ABI kernels
(include/sslrec_b200.h), written from the header's formulas rather than from the kernels, so the kernel tests
compare every launch variant with one plain statement of what it must compute.  No torch, no device.

  propagate_layer   ssl_propagate_layer (the formula block of the header: keep masks, edge_scale, in_views,
                    residual, noise, x_out, sum_out, reduce_views with the regulariser rows)
  rows_normalize    ssl_rows_normalize (rinv, the row-major copy, the K-major tile copy, the tf32 split)
  softmax_gemm_tiles  ssl_softmax_gemm / _tf32x3 per 64-column tile, so any n_split partition can be summed
  spmm_fma_chain    ssl_spmm_exact's documented order: one sequential fp32 FMA chain per output element
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from oracle import philox as P


# ---------------------------------------------------------------------------------------------------------------
# ssl_propagate_layer
# ---------------------------------------------------------------------------------------------------------------

def keep_masks(csr: dict, a: dict) -> list:
    """Per view: the effective weight multiplier m_v(p) * s_v of every CSR entry p (float64 [nnz]), and the bool keep
    mask.  edge_mode 0 keeps every entry at its stored value (edge_scale only scales kept entries of a masking view);
    mode 1 keeps iff U(seed, edge_stream_id, row, col) + keep >= 1 with (row, col) swapped when transpose; mode 2 reads
    edge_mask[p], or edge_mask[rev[p]] when transpose."""
    rows_g = np.repeat(csr['rows'], np.diff(csr['rowptr']))           # global row of every entry
    cols = csr['colidx'].astype(np.int64)
    out = []
    for v in range(a['n_views']):
        mode = a['edge_mode'][v]
        if mode == 0:
            keep = np.ones(cols.shape[0], dtype=bool)
            scale = 1.0
        elif mode == 1:
            kr, kc = (cols, rows_g) if a['transpose'] else (rows_g, cols)
            keep = P.edge_keep(a['seed'][v], a['edge_stream_id'], kr, kc, a['edge_keep'][v])
            scale = float(np.float32(a['edge_scale'][v]))
        else:
            m = np.asarray(a['edge_mask'][v])
            keep = (m[csr['rev']] if a['transpose'] else m) != 0
            scale = float(np.float32(a['edge_scale'][v]))
        out.append((keep, np.where(keep, scale, 0.0)))
    return out


def propagate_layer(csr: dict, a: dict, x_in: np.ndarray, residual=None, sum_src=(), reg_src=None, reg_src2=None, noise_u=None) -> dict:
    """One layer of ssl_propagate_layer in float64, for the rows the plan owns.

    csr: rowptr [n_local + 1], colidx / vals [nnz] (CSR of the owned rows, local order), rows [n_local] (global id of
         every local row), rev [nnz] or None, n (height of every table).
    a:   dim, n_views, in_views, transpose, reduce_views, sum_src_views, reg_coef, reg_coef_dev (float or None),
         edge_mode / edge_keep / edge_scale / edge_mask, noise_mode / noise_eps, seed, edge_stream_id, noise_stream_id
         (seed[v] is the seed the view actually uses).
    x_in [n, in_views, dim]; residual [n, V, dim]; sum_src[i] [n, sum_src_views[i], dim]; reg_src / reg_src2 [n, dim];
    noise_u[v] [n, dim] for noise_mode 2.
    Returns float64 arrays over the owned rows: x [n_local, V, dim] (the x_out rows), pre (x before the noise term),
    noise_abs (|noise term|), sum [n_local, V, dim] or [n_local, dim] with reduce_views, keep (per-view bool masks),
    and mag_x / mag_sum: the same sums over absolute values (the scale of the rounding error of an fp32 evaluation).
    """
    V, dim = a['n_views'], a['dim']
    n_loc = csr['rowptr'].shape[0] - 1
    g = csr['rows']
    x64 = np.asarray(x_in, dtype=np.float64)
    vals = csr['vals'].astype(np.float64)
    masks = keep_masks(csr, a)
    x = np.zeros((n_loc, V, dim))
    mag = np.zeros((n_loc, V, dim))
    for v in range(V):
        w = vals * masks[v][1]
        A = sp.csr_matrix((w, csr['colidx'].copy(), csr['rowptr'].copy()), shape=(n_loc, csr['n']))       # copies: scipy may
        Aa = sp.csr_matrix((np.abs(w), csr['colidx'].copy(), csr['rowptr'].copy()), shape=(n_loc, csr['n']))  # sort in place
        xv = x64[:, 0 if a['in_views'] == 1 else v, :]
        x[:, v] = A @ xv
        mag[:, v] = Aa @ np.abs(xv)
    if residual is not None:
        r = np.asarray(residual, dtype=np.float64)[g]
        x += r
        mag += np.abs(r)
    pre = x.copy()
    noise_abs = np.zeros_like(x)
    eps = float(np.float32(a['noise_eps']))
    for v in range(V):
        nm = a['noise_mode'][v]
        if nm == 0:
            continue
        if nm == 1:
            u = P.noise_uniform(a['seed'][v], a['noise_stream_id'], csr['n'], dim)[g].astype(np.float64)
        else:
            u = np.asarray(noise_u[v], dtype=np.float64)[g]
        d = eps * u / np.maximum(np.linalg.norm(u, axis=1, keepdims=True), 1e-12)
        x[:, v] += np.sign(pre[:, v]) * d
        noise_abs[:, v] = np.abs(d)
    mag_x = mag + noise_abs
    s, mag_s = x.copy(), mag_x.copy()
    for i, src in enumerate(sum_src):
        src = np.asarray(src, dtype=np.float64)[g]
        sv = a['sum_src_views'][i]
        t = src[:, [0] * V if sv == 1 else list(range(V)), :]
        s += t
        mag_s += np.abs(t)
    if a.get('reduce_views'):
        s, mag_s = s.sum(1), mag_s.sum(1)
        if reg_src is not None:
            c = float(np.float32(a['reg_coef'])) * (1.0 if a.get('reg_coef_dev') is None else float(np.float32(a['reg_coef_dev'])))
            t = c * np.asarray(reg_src, dtype=np.float64)[g]
            s += t
            mag_s += np.abs(t)
        if reg_src2 is not None:
            t = np.asarray(reg_src2, dtype=np.float64)[g]
            s += t
            mag_s += np.abs(t)
    return dict(x=x, pre=pre, noise_abs=noise_abs, sum=s, mag_x=mag_x, mag_sum=mag_s, keep=[m[0] for m in masks])


# ---------------------------------------------------------------------------------------------------------------
# ssl_rows_normalize and the tf32 split
# ---------------------------------------------------------------------------------------------------------------

def rows_normalize(x: np.ndarray, idx, norm_mode: int, alpha: float):
    """-> (out [n, dim], rinv [n]) in float64: row i is x[idx[i]] (idx None = identity) times rinv * alpha, with
    rinv = 1/sqrt(1e-8 + |x|^2) (mode 0), 1/max(|x + 1e-8|, 1e-12) applied to x + 1e-8 (mode 1), 1/max(|x|, 1e-12)
    (mode 2), 1 (mode 3)."""
    x = np.asarray(x, dtype=np.float64)
    if idx is not None:
        x = x[np.asarray(idx)]
    if norm_mode == 1:
        x = x + float(np.float32(1e-8))
    nrm = np.sqrt((x * x).sum(1))
    if norm_mode == 0:
        rinv = 1.0 / np.sqrt(float(np.float32(1e-8)) + nrm * nrm)
    elif norm_mode in (1, 2):
        rinv = 1.0 / np.maximum(nrm, float(np.float32(1e-12)))
    else:
        rinv = np.ones(x.shape[0])
    return x * rinv[:, None] * float(np.float32(alpha)), rinv


def k_major_tiles(out_padded: np.ndarray) -> np.ndarray:
    """The K-major tile copy [ceil(n/64), dim, 64] of a row-major [ceil64(n), dim] table: slot q of tile b holds row
    64 b + c with c = (q >> 2) + 16 (q & 3)."""
    n_pad, dim = out_padded.shape
    q = np.arange(64)
    c = (q >> 2) + 16 * (q & 3)
    t = out_padded.reshape(n_pad // 64, 64, dim)[:, c, :]          # [tiles, q, dim]
    return np.ascontiguousarray(t.transpose(0, 2, 1))


def tf32_rna(x: np.ndarray) -> np.ndarray:
    """cvt.rna.tf32.f32 on fp32 bits: round the 23-bit mantissa to 10 bits, to nearest with ties away from zero (add
    half a tf32 unit to the magnitude, clear the 13 low bits; a carry moves into the exponent).  Finite inputs."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_split(x: np.ndarray):
    """hi = tf32_rna(x), lo = tf32_rna(x - hi) (x - hi is exact in fp32)."""
    x = np.asarray(x, dtype=np.float32)
    hi = tf32_rna(x)
    return hi, tf32_rna((x - hi).astype(np.float32))


# ---------------------------------------------------------------------------------------------------------------
# ssl_softmax_gemm / ssl_softmax_gemm_tf32x3
# ---------------------------------------------------------------------------------------------------------------

def softmax_gemm_tiles(R: np.ndarray, C: np.ndarray, colscale, offset: float):
    """Per 64-column tile t of C: rowsum [n_tiles, n_r] = sum_c e, o [n_tiles, n_r, dim] = sum_c e C_c and the magnitude
    sum_c e |C_c|, with e = exp2(R_r . C_c - offset) * colscale[c], in float64 over columns [64 t, min(64 t + 64, n_c))."""
    R = np.asarray(R, dtype=np.float64)
    C = np.asarray(C, dtype=np.float64)
    n_c = C.shape[0]
    e = np.exp2(R @ C.T - float(np.float32(offset)))
    if colscale is not None:
        e = e * np.asarray(colscale, dtype=np.float64)[None, :n_c]
    n_t = (n_c + 63) // 64
    rs = np.stack([e[:, 64 * t:64 * t + 64].sum(1) for t in range(n_t)])
    o = np.stack([e[:, 64 * t:64 * t + 64] @ C[64 * t:64 * t + 64] for t in range(n_t)])
    mag = np.stack([e[:, 64 * t:64 * t + 64] @ np.abs(C[64 * t:64 * t + 64]) for t in range(n_t)])
    return rs, o, mag


def split_tiles(n_c: int, n_split: int):
    """The tile range [t0, t1) of each of the n_split chunks: t0 = n_ct * s / n_split (integer division)."""
    n_ct = (n_c + 63) // 64
    return [(n_ct * s // n_split, n_ct * (s + 1) // n_split) for s in range(n_split)]


# ---------------------------------------------------------------------------------------------------------------
# ssl_spmm_exact
# ---------------------------------------------------------------------------------------------------------------

def spmm_fma_chain(rowptr, colidx, vals, x: np.ndarray) -> np.ndarray:
    """y[r, j] = fma(w_e, x[col_e, j], acc) over the row's entries in CSR order from acc = 0, in fp32, emulated in float64
    (w * x of two floats is exact in double; the sum is rounded to double, then to float -- a double rounding that can
    differ from one fused rounding in the last bit, rarely)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    deg = np.diff(rowptr)
    x = np.asarray(x, dtype=np.float32)
    w = np.asarray(vals, dtype=np.float32).astype(np.float64)
    y = np.zeros((deg.shape[0], x.shape[1]), dtype=np.float32)
    for k in range(int(deg.max()) if deg.size else 0):
        rows = np.flatnonzero(deg > k)
        e = rowptr[rows] + k
        y[rows] = (w[e, None] * x[colidx[e]].astype(np.float64) + y[rows].astype(np.float64)).astype(np.float32)
    return y
