"""fp64 references of the learner's split-M weight-gradient reductions, chunk by chunk (test infrastructure).

Every reduction is dW[n, k] = sum_m dY[m, n] A[m, k] and dB[n] = sum_m dY[m, n] over the rows of a chunk,
[c * rpc, min((c + 1) * rpc, M)).  The operands are given as row-range functions `f(m0, m1) -> float64 [m1 - m0, cols]`
so that references past 2^24 rows are built slab by slab in float64 on the device.  Besides the sums, every reference
returns what the bars need: the sums of |dY[m, n] A[m, k]| and |dY[m, n]| (the element-wise error scale) and the sums
WITHOUT the last row of each chunk (to prove that the data makes a chunk's tail visible).
"""
import torch as th

F64 = th.float64


def n_chunks(M, rpc):
    return (M + rpc - 1) // rpc


def chunk_sums(dy_rows, a_rows, M, rpc, slab_rows=1 << 21):
    """Per-chunk fp64 sums of dY^T A: dict of W, W_abs, W_drop [nc, Nout, K] and B, B_abs, B_drop [nc, Nout]."""
    nc = n_chunks(M, rpc)
    L = min(rpc, M)                                   # every chunk but the last has rpc rows; the last is padded to L
    per = max(1, slab_rows // L)
    out = {k: [] for k in ("W", "W_abs", "W_drop", "B", "B_abs", "B_drop")}
    for c0 in range(0, nc, per):
        c1 = min(nc, c0 + per)
        m0, m1 = c0 * rpc, min(c1 * rpc, M)
        y, a = dy_rows(m0, m1), a_rows(m0, m1)
        pad = (c1 - c0) * L - (m1 - m0)
        if pad:
            y = th.cat([y, y.new_zeros(pad, y.shape[1])])
            a = th.cat([a, a.new_zeros(pad, a.shape[1])])
        y3, a3 = y.view(c1 - c0, L, -1), a.view(c1 - c0, L, -1)
        W = th.bmm(y3.transpose(1, 2), a3)
        B = y3.sum(1)
        last = th.tensor([min((c + 1) * rpc, M) - 1 - c * rpc for c in range(c0, c1)], device=y.device)
        ar = th.arange(c1 - c0, device=y.device)
        yl, al = y3[ar, last], a3[ar, last]
        out["W"].append(W)
        out["W_abs"].append(th.bmm(y3.abs().transpose(1, 2), a3.abs()))
        out["W_drop"].append(W - yl[:, :, None] * al[:, None, :])
        out["B"].append(B)
        out["B_abs"].append(y3.abs().sum(1))
        out["B_drop"].append(B - yl)
    return {k: th.cat(v) for k, v in out.items()}


def dense_rows(A, shift=0):
    """Rows of the dense loader: row m reads A[m - shift], zero for m < shift.  A: [rows, K] (any float dtype)."""
    def f(m0, m1):
        out = th.zeros(m1 - m0, A.shape[1], dtype=F64, device=A.device)
        lo = max(m0, shift)
        if lo < m1:
            out[lo - m0:] = A[lo - shift:m1 - shift].to(F64)
        return out
    return f


def state_rows(state, T, K, shift=0):
    """Rows of the state loader: row m = b*T + t reads state[b, t + shift, :K].  state: [B, TT, S]."""
    def f(m0, m1):
        m = th.arange(m0, m1, device=state.device)
        return state[m // T, m % T + shift, :K].to(F64)
    return f


def agent_rows(obs, onehot, last, aid):
    """Rows of the agent-input loader: row m = t*R + b*N + n reads [obs[b,t,n] | onehot[b,t-1,n] (zero at t = 0, present
    with last-action input) | e_n (present with agent-id input)].  obs [B,TT,N,OBS], onehot [B,TT,N,A]."""
    B, TT, N, OBS = obs.shape
    R = B * N

    def f(m0, m1):
        m = th.arange(m0, m1, device=obs.device)
        t, rr = m // R, m % R
        b, n = rr // N, rr % N
        parts = [obs[b, t, n].to(F64)]
        if last:
            prev = onehot[b, (t - 1).clamp_min(0), n].to(F64)
            parts.append(th.where((t > 0)[:, None], prev, 0.0))
        if aid:
            parts.append(th.nn.functional.one_hot(n, N).to(F64))
        return th.cat(parts, 1)
    return f


def gru_sums(x, hout, d_g, R, rpc):
    """k_reduce_gru: W_ih = d_g[:, :192]^T x, W_hh rows 0-127 = d_g[:, :128]^T h_prev, rows 128-191 = d_g[:, 192:]^T h_prev,
    h_prev[m] = hout[m - R] (zero for m < R); biases are the matching column sums.  Returns three chunk_sums dicts."""
    M1 = x.shape[0]
    cols = lambda lo, hi: (lambda m0, m1: d_g[m0:m1, lo:hi].to(F64))
    return (chunk_sums(cols(0, 192), dense_rows(x), M1, rpc),
            chunk_sums(cols(0, 128), dense_rows(hout, R), M1, rpc),
            chunk_sums(cols(192, 256), dense_rows(hout, R), M1, rpc))


def fc2_sums(d_chosen, actions, hout, A, grid):
    """k_fc2_grad over the T*R rows m = t*R + b*N + n: CTA c owns the rows with m mod (8 grid) in [8c, 8c + 8);
    W[c, a] = sum over its rows with action a of d_chosen[b,t,n] h[m], B[c, a] = sum d_chosen.  d_chosen [B,T,N],
    actions [B,TT,N,1] int64, hout [>= T*R, 64].  Returns the chunk_sums keys with W [grid, A, 64], B [grid, A]."""
    Bn, T, N = d_chosen.shape
    R = Bn * N
    rows = T * R
    m = th.arange(rows, device=hout.device)
    t, rr = m // R, m % R
    b, n = rr // N, rr % N
    d = d_chosen[b, t, n].to(F64)
    a = actions[b, t, n, 0]
    h = hout[:rows].to(F64)
    cta = (m % (8 * grid)) // 8
    key = cta * A + a
    out = {}
    for name, dv, hv in (("", d, h), ("_abs", d.abs(), h.abs())):
        out["W" + name] = th.zeros(grid * A, 64, dtype=F64, device=h.device).index_add_(0, key, dv[:, None] * hv).view(grid, A, 64)
        out["B" + name] = th.zeros(grid * A, dtype=F64, device=h.device).index_add_(0, key, dv).view(grid, A)
    lastrow = th.full((grid,), -1, dtype=th.long, device=h.device).scatter_reduce_(0, cta, m, "amax")
    W_drop, B_drop = out["W"].clone(), out["B"].clone()
    cs = th.nonzero(lastrow >= 0).flatten()                  # CTAs that own rows; each loses its last one
    r = lastrow[cs]
    W_drop[cs, a[r]] -= d[r, None] * h[r]
    B_drop[cs, a[r]] -= d[r]
    out["W_drop"], out["B_drop"] = W_drop, B_drop
    return out
